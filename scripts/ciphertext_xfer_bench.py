"""sunscreen Ciphertext bytes <-> device-resident ciphertexts: fhe_b200_upload_ciphertexts / fhe_b200_download_ciphertexts against
the host loop they replace.

For each batch size (host clock around the synchronous calls, after a warm-up, median of R repetitions):
  upload_seal        SEAL-written Ciphertexts (libzstd level 3, what the precompiles return by default) -> device words
  upload_structured  structured-writer Ciphertexts -> device words
  download_seal      device words -> Ciphertexts under the default writer (libzstd on the host cores)
  download_structured device words -> Ciphertexts under the structured writer (written on the GPU)
  base_upload_*      host loop of fhe_b200_parse_ciphertext into pinned memory + one H2D
  base_download_*    one D2H into pinned memory + host loop of fhe_b200_write_ciphertext
The ciphertexts are uniform random residues (their compression ratio is that of real encryptions).  Every result is checked:
uploaded words equal the source words, downloaded bytes equal the baseline's.  The GPU's name and power limit and the host's
core count are read in the same run.

  python scripts/ciphertext_xfer_bench.py [--sizes 256 4096 16384] [--reps 3] [--out result.json]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from fhe_precompiles_b200 import _lib, device  # noqa: E402

N = 4096
MODULI = (0xFFFFEE001, 0xFFFFC4001)
KIND = "i64"


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power, clock = (x.strip() for x in q.stdout.splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock, "torch_device": torch.cuda.get_device_name(0),
            "host_cores": os.cpu_count(), "host_cores_usable": len(os.sched_getaffinity(0))}


def median_s(fn, reps: int) -> float:
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return statistics.median(times)


def random_words(n: int, seed: int) -> torch.Tensor:
    g = torch.Generator(device="cuda").manual_seed(seed)
    ct = torch.empty((n, 2, 2, N), dtype=torch.int64, device="cuda")
    for limb, q in enumerate(MODULI):
        ct[:, :, limb, :] = torch.randint(0, q, (n, 2, N), dtype=torch.int64, device="cuda", generator=g)
    return ct


def set_writer(mode: int) -> None:
    _lib.lib().fhe_b200_set_zstd_writer(mode)


def base_upload(cts, pinned: torch.Tensor) -> torch.Tensor:
    L = _lib.lib()
    words = pinned[: len(cts)]
    base = words.data_ptr()
    for i, c in enumerate(cts):
        if L.fhe_b200_parse_ciphertext(c, len(c), base + i * 4 * N * 8, None, 0) != 0:
            raise RuntimeError("baseline parse failed")
    return words.to("cuda", non_blocking=True)


def base_download(ct: torch.Tensor, pinned: torch.Tensor, dt: bytes) -> list:
    L = _lib.lib()
    words = pinned[: ct.shape[0]]
    words.copy_(ct, non_blocking=True)
    torch.cuda.synchronize()
    out, out_len, res = ctypes.c_void_p(), ctypes.c_int64(), []
    base = words.data_ptr()
    for i in range(ct.shape[0]):
        if L.fhe_b200_write_ciphertext(base + i * 4 * N * 8, dt, ctypes.byref(out), ctypes.byref(out_len)) != 0:
            raise RuntimeError("baseline write failed")
        res.append(ctypes.string_at(out.value, out_len.value))
        L.fhe_free(out)
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 4096, 16384])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    device.init(0)
    info = gpu_info()
    print(json.dumps(info), flush=True)
    nmax = max(args.sizes)
    src = random_words(nmax, 1)
    prev = _lib.lib().fhe_b200_set_zstd_writer(-1)
    # the inputs: the library's own writers (byte-identical to what the precompiles return)
    set_writer(0)
    seal, st = device.download_ciphertexts(src, KIND)
    assert not st.any()
    set_writer(1)
    structured, st = device.download_ciphertexts(src, KIND)
    assert not st.any()
    dt = _dt_of(seal[0])
    pinned = torch.empty((nmax, 2, 2, N), dtype=torch.int64).pin_memory()
    rows = []
    for n in args.sizes:
        reps = args.reps
        r = {"n": n, "reps": reps}
        for name, cts in (("seal", seal[:n]), ("structured", structured[:n])):
            device.upload_ciphertexts(cts, KIND)  # warm-up
            d, st = device.upload_ciphertexts(cts, KIND)
            assert not st.any() and torch.equal(d, src[:n]), f"upload {name} {n}"
            r[f"upload_{name}_s"] = median_s(lambda: device.upload_ciphertexts(cts, KIND), reps)
            assert torch.equal(base_upload(cts, pinned), src[:n])
            r[f"base_upload_{name}_s"] = median_s(lambda: base_upload(cts, pinned), reps if n <= 4096 else 1)
        for mode, name in ((0, "seal"), (1, "structured")):
            set_writer(mode)
            out, st = device.download_ciphertexts(src[:n], KIND)
            assert not st.any() and out == (seal if mode == 0 else structured)[:n], f"download {name} {n}"
            r[f"download_{name}_s"] = median_s(lambda: device.download_ciphertexts(src[:n], KIND), reps)
            ref = base_download(src[: min(n, 256)], pinned, dt)
            assert ref == out[: len(ref)], f"baseline download {name}"
            r[f"base_download_{name}_s"] = median_s(lambda: base_download(src[:n], pinned, dt), reps if n <= 4096 else 1)
        for k in [k for k in r if k.endswith("_s")]:
            r[k[:-2] + "_us_per_ct"] = round(r[k] / n * 1e6, 2)
            r[k[:-2] + "_k_per_s"] = round(n / r[k] / 1e3, 2)
            r[k] = round(r[k], 5)
        rows.append(r)
        print(json.dumps(r), flush=True)
    _lib.lib().fhe_b200_set_zstd_writer(prev)
    res = dict(info, kind=KIND, rows=rows)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


def _dt_of(ct: bytes) -> bytes:
    n = int.from_bytes(ct[:8], "little")
    return ct[8 : 8 + n]


if __name__ == "__main__":
    main()
