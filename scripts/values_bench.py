"""Device-resident typed values: time of encode / decode, and what they add to encrypt / decrypt_checked.

For each kind and batch size (CUDA events, after warm-up, R repetitions; the A/B pairs alternate within each repetition):
  encode, decode                               ms per call, M ops/s, bytes per op the kernel must move, GB/s
  encrypt_values     against encrypt           on the same values / pre-encoded plaintexts
  decrypt_values     against decrypt_checked   on the same ciphertexts
frac64 decode is timed on realistic plaintexts (decryptions of mul_relin products) and on dense uniform uint16 rows, the worst
case of its in-order sum.  Every input is at least 134 MB (plaintexts) or 1 GB (ciphertexts), past the 126 MB L2.  The GPU's
name and power limit are read in the same run and printed with the numbers.

  python scripts/values_bench.py [--sizes 16384 65536] [--reps 10] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from fhe_precompiles_b200 import _lib, device  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 4096
# bytes the kernels have to move per op: encode writes the 8 KB row (reads the value); integer decode reads the 64 / 256
# coefficients the decoder uses; frac64 decode reads coefficients 0..63 and 3016..4095 (below index 3022 every term is 0)
ENC_BYTES = {"u256": 2 * N + 32, "u64": 2 * N + 8, "i64": 2 * N + 8, "frac64": 2 * N + 8}
DEC_BYTES = {"u256": 2 * 256 + 32, "u64": 2 * 64 + 8, "i64": 2 * 64 + 8, "frac64": 2 * (64 + 1080) + 8}


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power, clock = (x.strip() for x in q.stdout.splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock, "torch_device": torch.cuda.get_device_name(0)}


def timed(fns, reps: int, warmup: int = 3) -> list:
    """ms per call of each fn, the fns alternating within every repetition"""
    for _ in range(warmup):
        for f in fns:
            f()
    total = [0.0] * len(fns)
    for _ in range(reps):
        for k, f in enumerate(fns):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            total[k] += e0.elapsed_time(e1)
    return [t / reps for t in total]


def random_values(kind: str, n: int, g: torch.Generator) -> torch.Tensor:
    if kind == "frac64":
        mant = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
        return mant * torch.pow(10.0, torch.randint(-12, 12, (n,), device="cuda", generator=g).double())
    shape = (n, 4) if kind == "u256" else (n,)
    return torch.randint(-(2**63), 2**63 - 1, shape, dtype=torch.int64, device="cuda", generator=g)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[16384, 65536])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    device.init(0)
    pk, rk = device.parse_public_key(open(os.path.join(ROOT, "fhe_precompiles_b200/data/network.pub"), "rb").read())
    pri = open(os.path.join(ROOT, "fhe_precompiles_b200/data/network.pri"), "rb").read()
    sk = torch.empty((3, N), dtype=torch.int64)
    assert _lib.lib().fhe_b200_parse_private_key(pri, len(pri), sk.data_ptr()) == 0
    pk, rk, sk = pk.cuda(), rk.cuda(), sk.cuda()
    g = torch.Generator(device="cuda").manual_seed(1)
    result = {**gpu_info(), "reps": args.reps, "rows": []}
    for n in args.sizes:
        seeds = torch.randint(-(2**63), 2**63 - 1, (n, 8), dtype=torch.int64, device="cuda", generator=g)
        dense = torch.randint(-(2**15), 2**15, (n, N), dtype=torch.int16, device="cuda", generator=g)
        for kind in device.VALUE_KINDS:
            values = random_values(kind, n, g)
            plain, status = device.encode(kind, values)
            assert not status.any().item()
            assert torch.equal(device.decode(kind, plain), values), kind  # round trip of in-range values
            ct = device.encrypt(pk, plain, seeds)
            row = {"kind": kind, "n": n}
            (enc_ms,) = timed([lambda: device.encode(kind, values)], args.reps)
            row["encode_ms"], row["encode_mops"] = round(enc_ms, 4), round(n / enc_ms / 1e3, 2)
            row["encode_gbs"] = round(n * ENC_BYTES[kind] / enc_ms / 1e6, 1)
            e_ms, ev_ms = timed([lambda: device.encrypt(pk, plain, seeds), lambda: device.encrypt_values(pk, kind, values, seeds)], args.reps)
            row["encrypt_ms"], row["encrypt_values_ms"] = round(e_ms, 3), round(ev_ms, 3)
            row["encrypt_values_overhead_pct"] = round(100 * (ev_ms / e_ms - 1), 2)
            d_ms, dv_ms = timed([lambda: device.decrypt_checked(ct, sk), lambda: device.decrypt_values(ct, sk, kind)], args.reps)
            row["decrypt_checked_ms"], row["decrypt_values_ms"] = round(d_ms, 3), round(dv_ms, 3)
            row["decrypt_values_overhead_pct"] = round(100 * (dv_ms / d_ms - 1), 2)
            real = device.decrypt(device.mul_relin(ct, ct, rk), sk)  # decrypted products: a chain's realistic last plaintexts
            inputs = {"decode_real": real, "decode_dense": dense} if kind == "frac64" else {"decode_real": real}
            for name, p in inputs.items():
                (ms,) = timed([lambda: device.decode(kind, p)], args.reps)
                row[name + "_ms"], row[name + "_mops"] = round(ms, 4), round(n / ms / 1e3, 2)
                row[name + "_gbs"] = round(n * DEC_BYTES[kind] / ms / 1e6, 1)
            del ct, real
            result["rows"].append(row)
            print(json.dumps(row), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != "rows"}))


if __name__ == "__main__":
    main()
