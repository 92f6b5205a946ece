"""Multiply + relinearise under many users' keys: fhe_b200_batch of mul_cipheri64_cipheri64 under 1, 16 and 256 distinct user
keys at 256, 4,096 and 16,384 calls, under both result writers; and, device-resident at n = 4,096, mul_relin_keyed with 1, 64
and 4,096 keys against mul_relin under one key and against K separate mul_relin calls of n / K rows each.

    python scripts/multikey_batch_bench.py --out profiles/multikey_batch.json [--package-root DIR] [--label NAME]

--package-root imports fhe_precompiles_b200 from another tree (e.g. a build of an earlier commit) so that two versions can be
measured alternately in one session; a tree without mul_relin_keyed measures the rest.  User keys are the fixture key with
seeded uniform relinearisation keys (tests/user_keys.py).  Operands are 256 distinct libzstd-written i64 ciphertexts (the
library's own encrypt_i64); call i uses key i mod K, so the calls of one key are spread over the batch as a block's are.  A
byte-surface point is the median of --reps (default 3) timed batches after one warm-up batch of the same calls; a device point
is the median of --reps CUDA-event timings of --iters back-to-back calls after one warm-up.  The GPU's name and power limit and
the host's core count are recorded with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 4096


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (x.strip() for x in q.stdout.splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "host_cores_usable": len(os.sched_getaffinity(0))}


def byte_surface(args, FHE, L, pack, users) -> list:
    distinct = 256
    prev = L.fhe_b200_set_zstd_writer(0)
    cts = FHE.run_batch([("encrypt_i64", pack.pack_two_arguments(pack.serialize_i64(i * 7919 - 10**6), i.to_bytes(4, "big")))
                         for i in range(distinct)])
    assert all(st == 0 for st, _ in cts)
    cts = [ct for _, ct in cts]
    rows = []
    try:
        for writer in (0, 1):
            L.fhe_b200_set_zstd_writer(writer)
            for k in (int(x) for x in args.keys.split(",")):
                packed = [pack.pack_binary_operation(users[i % k][0], cts[i % distinct], cts[(i + 1) % distinct])
                          for i in range(max(distinct, k))]
                for n in (int(x) for x in args.sizes.split(",")):
                    calls = [("mul_cipheri64_cipheri64", packed[i % len(packed)]) for i in range(n)]
                    res = FHE.run_batch(calls)  # warm-up: lanes, staging and key cache at this size
                    failed = sum(1 for st, _ in res if st)
                    del res
                    times = []
                    for _ in range(args.reps):
                        t0 = time.perf_counter()
                        FHE.run_batch(calls)
                        times.append(time.perf_counter() - t0)
                    t = statistics.median(times)
                    rows.append({"writer": "structured" if writer else "seal", "keys": k, "calls": n, "seconds": t,
                                 "calls_per_s": n / t, "failed": failed, "seconds_each": times})
                    print(f"{args.label:>12} {rows[-1]['writer']:>10} keys {k:>4} {n:>6}: {n / t:>10.0f} calls/s", flush=True)
    finally:
        L.fhe_b200_set_zstd_writer(prev)
    return rows


def device_resident(args, device, users) -> list:
    import torch

    n = args.device_n
    rng = np.random.default_rng(4)
    moduli = (0xFFFFEE001, 0xFFFFC4001)
    ct = np.empty((2, n, 2, 2, N), dtype=np.uint64)
    for l, q in enumerate(moduli):
        ct[:, :, :, l, :] = rng.integers(0, q, size=(2, n, 2, N), dtype=np.uint64)
    a, b = (torch.from_numpy(x.view(np.int64)).cuda() for x in ct)
    out = torch.empty_like(a)
    key_moduli = (0xFFFFEE001, 0xFFFFC4001, 0x1FFFFE0001)
    kmax = max(int(x) for x in args.device_keys.split(","))
    rks_h = np.empty((kmax, 2, 2, 3, N), dtype=np.uint64)
    rks_h[: len(users)] = np.stack([rk for _, rk in users])[:kmax]
    for l, q in enumerate(key_moduli):  # beyond the byte-surface users: seeded uniform keys of the same form
        rks_h[len(users):, :, :, l, :] = rng.integers(0, q, size=(max(0, kmax - len(users)), 2, 2, N), dtype=np.uint64)
    rks = torch.from_numpy(rks_h.view(np.int64)).cuda()
    keyed = hasattr(device, "mul_relin_keyed")

    def timed(fn) -> tuple:
        fn()  # warm-up: scratch arena, key preparation buffers
        torch.cuda.synchronize()
        times = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                fn()
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1) / args.iters)
        return statistics.median(times), times

    rows = []

    def add(name, k, fn):
        ms, each = timed(fn)
        rows.append({"variant": name, "keys": k, "n": n, "ms": ms, "ops_per_s": n / ms * 1e3, "ms_each": each})
        print(f"{args.label:>12} device {name:>18} K {k:>5}: {ms:8.3f} ms  {n / ms * 1e3:>10.0f} ops/s", flush=True)

    add("mul_relin", 1, lambda: device.mul_relin(a, b, rks[0], out))
    for k in (int(x) for x in args.device_keys.split(",")):
        if keyed:
            idx = torch.from_numpy((np.arange(n) % k).astype(np.int32)).cuda()
            ks = rks[:k].contiguous()
            add("mul_relin_keyed", k, lambda: device.mul_relin_keyed(a, b, ks, idx, out))
        if k > 1:
            rows_per = n // k  # what a caller without keyed calls does: one call per key over that key's rows
            parts = [(a[j * rows_per:(j + 1) * rows_per], b[j * rows_per:(j + 1) * rows_per], rks[j], out[j * rows_per:(j + 1) * rows_per])
                     for j in range(k)]
            add("mul_relin_per_key", k, lambda: [device.mul_relin(x, y, r, o) for x, y, r, o in parts])
    return rows


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--package-root", default=ROOT)
    ap.add_argument("--label", default="this tree")
    ap.add_argument("--sizes", default="256,4096,16384")
    ap.add_argument("--keys", default="1,16,256")
    ap.add_argument("--device-n", type=int, default=4096)
    ap.add_argument("--device-keys", default="1,64,4096")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()
    sys.path[:0] = [args.package_root, os.path.join(ROOT, "tests"), ROOT]
    from fhe_precompiles_b200 import FHE, _lib, device, pack
    from user_keys import user_keys

    device.init(0)
    L = _lib.lib()
    users = user_keys(max(int(x) for x in args.keys.split(",")))
    out = {"label": args.label, "package_root": os.path.relpath(args.package_root, ROOT), "reps": args.reps,
           "statistic": "median of the timed batches (byte surface) or of the CUDA-event timings of --iters calls (device)",
           **gpu_info(), "device": device_resident(args, device, users), "byte_surface": byte_surface(args, FHE, L, pack, users)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
