"""Device zstd inflate (fhe_b200_zstd_inflate) against libzstd: ciphertext-payload-sized frames of several kinds and levels,
corrupted frames, and the kernel's throughput.  Needs a GPU."""
import ctypes
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fhe_precompiles_b200 import _lib  # noqa: E402
from oracle import formats as F  # noqa: E402  (checker only)

PAYLOAD = 131169


def inflate(L, frames):
    n = len(frames)
    bufs = [ctypes.create_string_buffer(f, len(f)) for f in frames]
    ptrs = (ctypes.c_void_p * n)(*[ctypes.cast(b, ctypes.c_void_p) for b in bufs])
    lens = (ctypes.c_size_t * n)(*[len(f) for f in frames])
    out = ctypes.create_string_buffer(n * PAYLOAD)
    status = (ctypes.c_int32 * n)()
    ms = ctypes.c_float()
    rc = L.fhe_b200_zstd_inflate(0, ptrs, lens, n, out, status, ctypes.byref(ms))
    assert rc == 0, L.fhe_b200_last_error()
    raw = out.raw  # one copy (out.raw copies the whole buffer every time it is evaluated)
    return [raw[i * PAYLOAD : (i + 1) * PAYLOAD] for i in range(n)], list(status), ms.value


def main() -> None:
    L = _lib.lib()
    z = F.zstd()
    rng = np.random.default_rng(11)
    q = (0xFFFFEE001, 0xFFFFC4001)
    prefix = bytes(rng.integers(0, 256, 97, dtype=np.uint8))

    def ct_payload():
        return prefix + np.stack([rng.integers(0, q[l], 4096, dtype=np.uint64) for _ in range(2) for l in range(2)]).tobytes()

    payloads, frames = [], []
    for lvl in (-3, 1, 3, 3, 3, 7, 12, 19):
        p = ct_payload()
        payloads.append(p), frames.append(z.compress(p, lvl))
    for kind in range(4):  # other content of the same size: text-like (Huffman literals), sparse, constant, random
        if kind == 0:
            p = bytes(rng.choice(list(b"abcdefgh \n"), size=PAYLOAD).astype(np.uint8))
        elif kind == 1:
            p = (rng.integers(0, 256, PAYLOAD, dtype=np.uint8) & rng.integers(0, 256, PAYLOAD, dtype=np.uint8) & rng.integers(0, 256, PAYLOAD, dtype=np.uint8)).tobytes()
        elif kind == 2:
            p = bytes(PAYLOAD)
        else:
            p = rng.integers(0, 256, PAYLOAD, dtype=np.uint8).tobytes()
        for lvl in (1, 3, 19):
            payloads.append(p), frames.append(z.compress(p, lvl))
    payloads.append(payloads[0]), frames.append(F.zstd_structured_frame(payloads[0]))
    got, status, _ = inflate(L, frames)
    ok = sum(1 for s in status if s == 1)
    for i, (g, w, s) in enumerate(zip(got, payloads, status)):
        assert s in (1, 2)
        if s == 1:
            assert g == w, f"frame {i}: device inflate differs from libzstd"
    # corrupted frames: never "ok" with different bytes than libzstd
    bad_frames, wants = [], []
    for it in range(96):
        fr = bytearray(frames[it % 8])
        k = it % 3
        if k == 0:
            fr[rng.integers(0, len(fr))] ^= 1 << rng.integers(0, 8)
        elif k == 1:
            fr = fr[: rng.integers(1, len(fr))]
        else:
            i = rng.integers(0, len(fr) - 4)
            fr[i : i + 4] = bytes(rng.integers(0, 256, 4, dtype=np.uint8))
        bad_frames.append(bytes(fr))
        try:
            wants.append(z.decompress(bytes(fr)) if z.lib.ZSTD_getFrameContentSize(bytes(fr), len(fr)) == PAYLOAD else None)
        except Exception:  # noqa: BLE001
            wants.append(None)
    got_b, status_b, _ = inflate(L, bad_frames)
    for g, w, s in zip(got_b, wants, status_b):
        if s == 1:
            assert w is not None and g == w, "device inflate accepted a frame libzstd rejects or decodes differently"
    # throughput: many level-3 ciphertext frames at once
    many = [z.compress(ct_payload(), 3) for _ in range(64)]
    res = {"valid_frames": len(frames), "valid_ok": ok, "corrupted_ok_and_equal": sum(1 for s in status_b if s == 1)}
    for n in (1, 64, 1024, 4096):
        fs = [many[i % 64] for i in range(n)]
        _, st, ms = inflate(L, fs)
        assert all(s == 1 for s in st)
        res[f"inflate_{n}_frames_ms"] = round(ms, 3)
        res[f"inflate_{n}_frames_per_s"] = round(n / (ms * 1e-3))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
