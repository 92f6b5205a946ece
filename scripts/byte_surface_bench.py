"""Byte-surface throughput of a LARGE batch (fhe_b200_batch, mul_cipheri64_cipheri64, operands as SEAL writes them: libzstd level-3
frames; every call carries its own copy of the public key) by batch size and result writer (FHE_B200_ZSTD_WRITER).  Below 2,048
calls the batch runs in 16-call tiles whose operands the host inflates, from 2,048 on in big tiles whose operands the GPU
inflates.  Every configuration runs in its own process:
    python scripts/byte_surface_bench.py                      # sweep (parent)
    python scripts/byte_surface_bench.py child <calls>        # one configuration, writer from the environment
Checks the first and last results against the single-call symbol."""
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def child(n: int, distinct: int = int(os.environ.get("BSB_DISTINCT", "256"))) -> None:
    from fhe_precompiles_b200 import FHE, _lib, pack

    L = _lib.lib()
    rng = np.random.default_rng(3)
    q = (0xFFFFEE001, 0xFFFFC4001)
    dt = b"sunscreen::types::bfv::signed::Signed,0.8.1,true"

    def blob() -> bytes:
        w = np.stack([rng.integers(0, q[l], 4096, dtype=np.uint64) for _ in range(2) for l in range(2)]).reshape(-1)
        out, ln = ctypes.c_void_p(), ctypes.c_int64()
        assert L.fhe_b200_write_ciphertext(w.ctypes.data, dt, ctypes.byref(out), ctypes.byref(ln)) == 0
        b = ctypes.string_at(out.value, ln.value)
        L.fhe_free(out)
        return b

    net_pub = FHE.public_key_bytes(b"")
    prev = L.fhe_b200_set_zstd_writer(0)
    packed = [pack.pack_binary_operation(net_pub, blob(), blob()) for _ in range(distinct)]
    L.fhe_b200_set_zstd_writer(prev)
    bufs = [(ctypes.c_char * len(p)).from_buffer_copy(p) for p in packed]
    op = L.fhe_b200_op_index(b"mul_cipheri64_cipheri64")
    arr = (_lib.BatchCall * n)()
    for i in range(n):
        arr[i].op, arr[i].bytes, arr[i].bytes_length = op, ctypes.cast(bufs[i % distinct], ctypes.c_void_p), len(packed[i % distinct])
    want = {k: FHE.mul_cipheri64_cipheri64(packed[k % distinct]) for k in (0, n - 1)}
    rates = []
    for rep in range(5):
        t0 = time.perf_counter()
        failed = L.fhe_b200_batch(arr, n, 0)
        dt_ = time.perf_counter() - t0
        assert failed == 0, failed
        for k, w in want.items():
            assert ctypes.string_at(arr[k].output, arr[k].output_length) == w, "batch result differs from the single call"
        for i in range(n):
            L.fhe_free(arr[i].output)
        rates.append(n / dt_)
    writer = os.environ.get("FHE_B200_ZSTD_WRITER", "default")
    print(json.dumps({"calls": n, "cores": os.cpu_count(), "FHE_B200_ZSTD_WRITER": writer, "calls_per_s_by_rep": [round(r) for r in rates], "best": round(max(rates[1:]))}),
          flush=True)


def main() -> None:
    if len(sys.argv) > 1 and sys.argv[1] == "child":
        child(int(sys.argv[2]))
        return
    sweeps = [(n, {"FHE_B200_ZSTD_WRITER": w}) for w in ("0", "1") for n in (1024, 2048, 4096, 8192)]
    for n, env in sweeps:
        e = dict(os.environ)
        e.update(env)
        e.setdefault("FHE_B200_QUIET", "1")
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "child", str(n)], env=e, capture_output=True, text=True, timeout=900)
        print(r.stdout.strip() or ("FAILED " + json.dumps(env) + " " + r.stderr[-600:]), flush=True)


if __name__ == "__main__":
    main()
