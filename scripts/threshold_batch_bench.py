"""Calls per second of fhe_b200_batch on the threshold precompiles: batches of 256, 4,096 and 16,384 calls of encrypt_i64,
decrypt_i64, reencrypt_i64 and of a mix of the three, under both result writers.

    python scripts/threshold_batch_bench.py --out profiles/threshold_batch.json [--package-root DIR] [--label NAME]

--package-root imports fhe_precompiles_b200 from another tree (e.g. a build of an earlier commit) so that two versions can
be measured alternately in one session.  Decrypt operands are libzstd-written ciphertexts (what SEAL and the default writer
produce), made by the library's own encrypt_i64; re-encryptions go to tests/data/public_key.bin.  Operand bytes cycle through
256 distinct inputs (a re-encryption input carries a ~400 KB public key): the library caches no results, so every call does
its full work.  Each point is the median of --reps (default 3) timed batches after one warm-up batch of the same size.  The GPU's name
and power limit and the host's core count are recorded with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (x.strip() for x in q.stdout.splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "host_cores_usable": len(os.sched_getaffinity(0))}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--package-root", default=ROOT)
    ap.add_argument("--label", default="this tree")
    ap.add_argument("--sizes", default="256,4096,16384")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    sys.path.insert(0, args.package_root)
    from fhe_precompiles_b200 import FHE, _lib, pack

    L = _lib.lib()
    pub = open(os.path.join(ROOT, "tests/data/public_key.bin"), "rb").read()
    distinct = 256
    enc_in = [pack.pack_two_arguments(pack.serialize_i64(i * 7919 - 10**6), i.to_bytes(4, "big")) for i in range(distinct)]
    prev = L.fhe_b200_set_zstd_writer(0)
    cts = FHE.run_batch([("encrypt_i64", x) for x in enc_in])
    assert all(st == 0 for st, _ in cts)
    cts = [ct for _, ct in cts]
    re_in = [pack.pack_binary_operation(pub, ct, b"bench %d" % i) for i, ct in enumerate(cts)]
    workloads = {
        "encrypt": lambda i: ("encrypt_i64", enc_in[i % distinct]),
        "decrypt": lambda i: ("decrypt_i64", cts[i % distinct]),
        "reencrypt": lambda i: ("reencrypt_i64", re_in[i % distinct]),
        "mix": lambda i: (("encrypt_i64", enc_in[i // 3 % distinct]), ("decrypt_i64", cts[i // 3 % distinct]),
                          ("reencrypt_i64", re_in[i // 3 % distinct]))[i % 3],
    }
    rows = []
    try:
        for writer in (0, 1):
            L.fhe_b200_set_zstd_writer(writer)
            for name, make in workloads.items():
                for n in (int(x) for x in args.sizes.split(",")):
                    calls = [make(i) for i in range(n)]
                    res = FHE.run_batch(calls)  # warm-up: lanes, staging and key cache at this size
                    failed = sum(1 for st, _ in res if st)
                    del res
                    times = []
                    for _ in range(args.reps):
                        t0 = time.perf_counter()
                        FHE.run_batch(calls)
                        times.append(time.perf_counter() - t0)
                    t = statistics.median(times)
                    rows.append({"writer": "structured" if writer else "seal", "workload": name, "calls": n, "seconds": t,
                                 "calls_per_s": n / t, "failed": failed, "seconds_each": times})
                    print(f"{args.label:>12} {rows[-1]['writer']:>10} {name:>9} {n:>6}: {n / t:>10.0f} calls/s", flush=True)
    finally:
        L.fhe_b200_set_zstd_writer(prev)
    out = {"label": args.label, "package_root": os.path.relpath(args.package_root, ROOT), "reps": args.reps,
           "statistic": "median of the timed batches, after one warm-up batch", **gpu_info(), "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
