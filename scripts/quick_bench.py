"""Scratch timing of the device-resident kernels (CUDA events). Not the contract bench (see bench.py)."""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from fhe_precompiles_b200 import device  # noqa: E402
from helpers import MODULI, N, KeySet, random_ct  # noqa: E402


def timeit(fn, iters=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
    ev[0].record()
    for i in range(iters):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    return min(ev[i].elapsed_time(ev[i + 1]) for i in range(iters))


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    device.init(0)
    keys = KeySet.load()
    rng = np.random.default_rng(0)
    base = random_ct(rng, 64)
    reps = (n + 63) // 64
    a = torch.from_numpy(np.tile(base, (reps, 1, 1, 1))[:n].view(np.int64)).cuda()
    b = torch.from_numpy(np.tile(base[::-1], (reps, 1, 1, 1))[:n].view(np.int64).copy()).cuda()
    rk = torch.from_numpy(keys.rk.view(np.int64)).cuda()
    out = torch.empty_like(a)
    ms = timeit(lambda: device.mul_relin(a, b, rk, out=out))
    print(f"mul_relin n={n}: {ms:.3f} ms  -> {n / ms * 1e3:.0f} ops/s")
    device.set_kernel_timing(True)
    device.mul_relin(a, b, rk, out=out)
    rep = device.kernel_timing_report(0)
    device.set_kernel_timing(False)
    print("   ", {k: round(v[0] / n * 1e3, 3) for k, v in rep.items()}, "us/op")
    c3 = device.multiply(a, b)
    ms = timeit(lambda: device.relinearize(c3, rk))
    print(f"  relinearize: {ms:.3f} ms ({ms / n * 1e3:.2f} us/op)")
    ms = timeit(lambda: device.add(a, b))
    print(f"  add:         {ms:.3f} ms  -> {n * 393216 / ms / 1e6:.0f} GB/s")
    pl = torch.randint(0, 4096, (n, N), dtype=torch.int16, device="cuda")
    ms = timeit(lambda: device.plain_addsub(a, pl, 0))
    print(f"  add_plain:   {ms:.3f} ms  -> {n * (2 * 131072 + 8192) / ms / 1e6:.0f} GB/s, {n / ms * 1e3 / 1e6:.2f} M ops/s")
    ms = timeit(lambda: device.multiply_plain(a, pl))
    print(f"  mul_plain:   {ms:.3f} ms  ({ms / n * 1e3:.3f} us/op) -> {n / ms * 1e3 / 1e6:.2f} M ops/s")
    for m in (0, 3):
        x = torch.from_numpy(rng.integers(0, MODULI[m], size=(n * 4, N), dtype=np.uint64).view(np.int64)).cuda()
        ms = timeit(lambda: device.ntt_(x, [m]))
        print(f"  ntt mod{m} x{n*4}: {ms:.3f} ms -> {n * 4 / ms * 1e3 / 1e6:.2f} M limb-NTT/s, {n*4*65536/ms/1e6:.0f} GB/s")
        ms = timeit(lambda: device.ntt_(x, [m], inverse=True))
        print(f"  intt mod{m} x{n*4}: {ms:.3f} ms -> {n * 4 / ms * 1e3 / 1e6:.2f} M limb-NTT/s")


if __name__ == "__main__":
    main()
