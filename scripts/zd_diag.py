"""Device zstd inflate timing (fhe_b200_zstd_inflate): ciphertext, text and structured frames, and batches of 32 to 8,192
level-3 ciphertext frames."""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import zstd_device_check as Z
from fhe_precompiles_b200 import _lib
from oracle import formats as F
L = _lib.lib(); z = F.zstd(); rng = np.random.default_rng(1)
q = (0xFFFFEE001, 0xFFFFC4001)
def ct(): return bytes(97) + np.stack([rng.integers(0, q[l], 4096, dtype=np.uint64) for _ in range(2) for l in range(2)]).tobytes()
def run(tag, frames, payloads):
    got, st, ms = Z.inflate(L, frames)
    ok = all((s != 1) or g == p for g, p, s in zip(got, payloads, st))
    print(tag, "ok", sum(1 for s in st if s == 1), "/", len(st), "kernel_ms", round(ms, 2), "frames/s", round(len(frames) / (ms * 1e-3)), "match", ok, flush=True)
p = ct()
cts = [ct() for _ in range(16)]
frs = [z.compress(c, 3) for c in cts]
t = bytes(rng.choice(list(b"abcdefgh \n"), size=Z.PAYLOAD).astype(np.uint8))
run("warm", [frs[0]], [cts[0]])
run("ct_l3 x1", [frs[0]], [cts[0]])
run("text_l3 x1", [z.compress(t, 3)], [t])
run("structured x1", [F.zstd_structured_frame(cts[0])], [cts[0]])
for n in (32, 256, 1024, 4096, 8192):
    run(f"ct_l3 x{n}", [frs[i % 16] for i in range(n)], [cts[i % 16] for i in range(n)])
