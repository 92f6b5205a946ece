"""The device zstd decoder's source (csrc/zstd_dec.h, zstd_plan2.h, zstd_exec3.h), built for the host by tests/zd_host.cpp,
against libzstd: every fixture blob of the reference (written by SEAL's bundled zstd 1.4.x, including Huffman, treeless and
repeat-mode blocks), random data of many shapes at many levels, structured frames, and mutated frames.  Contract under test:
status 0 => bytes identical to libzstd's; anything else is a hand-back to the host (status 1), never a wrong answer.  CPU only."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from helpers import ROOT
from oracle import formats as F


@pytest.fixture(scope="module")
def zd(tmp_path_factory):
    out = tmp_path_factory.mktemp("zd") / "libzd_host.so"
    src = os.path.join(ROOT, "tests", "zd_host.cpp")
    inc = os.path.join(ROOT, "fhe_precompiles_b200", "csrc")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I" + inc, src, "-o", str(out)], check=True)
    lib = ctypes.CDLL(str(out))
    cap = 1 << 21
    buf = ctypes.create_string_buffer(cap)
    fn = lib.zd_decode
    fn.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t),
                   ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_long)]

    def decode(frame: bytes):
        n, rounds, polls = ctypes.c_size_t(), ctypes.c_int(), ctypes.c_long()
        rc = fn(frame, len(frame), buf, cap, ctypes.byref(n), ctypes.byref(rounds), ctypes.byref(polls))
        assert rc != 2, "the parallel executor's copy phase stopped making progress"
        decode.rounds, decode.polls = rounds.value, polls.value
        return rc, (buf.raw[: n.value] if rc == 0 else None)

    decode.max_content = 131169  # one ciphertext payload: what k_zd3_exec holds in shared memory
    return decode


def _reference(frame: bytes):
    z = F.zstd()
    try:
        if z.lib.ZSTD_getFrameContentSize(frame, len(frame)) > (1 << 21):
            return None
        return z.decompress(frame)
    except ValueError:
        return None


def _frame_in(blob: bytes) -> bytes:
    assert blob[5] == F.COMPR_ZSTD
    return blob[16:]


def test_reference_fixtures_decode_identically(zd):
    frames = []
    for path in ("fhe_precompiles_b200/data/network.pub", "tests/data/public_key.bin"):
        pk = F.PublicKey.from_bytes(open(os.path.join(ROOT, path), "rb").read())
        frames += [_frame_in(pk.public_key.blob), _frame_in(pk.relin_key.blob)]
    for path in ("fhe_precompiles_b200/data/network.pri", "tests/data/private_key.bin"):
        frames.append(_frame_in(F.WithContext.read(F.Reader(open(os.path.join(ROOT, path), "rb").read())).blob))
    for path in ("tests/golden/ct_i64_16_seed11.bin", "tests/golden/ct_i64_mul_16_4.bin"):
        r = F.Reader(open(os.path.join(ROOT, path), "rb").read())
        r.take(r.u64()), r.u32(), r.u64()
        frames.append(_frame_in(F.WithContext.read(r).blob))
    for fr in frames:
        rc, got = zd(fr)
        want = F.zstd().decompress(fr)
        if len(want) > zd.max_content:
            assert rc == 1  # (keys: the parallel executor holds one ciphertext payload)
            continue
        assert rc == 0 and got == want


def _samples(rng):
    q = (0xFFFFEE001, 0xFFFFC4001)
    yield b"\0" * 97 + np.stack([rng.integers(0, q[l], 4096, dtype=np.uint64) for _ in range(2) for l in range(2)]).tobytes()
    yield bytes(rng.choice(list(b"abcdefgh \n"), size=int(rng.integers(1, 200000))).astype(np.uint8))
    yield rng.integers(0, 256, int(rng.integers(0, 5000)), dtype=np.uint8).tobytes()
    yield bytes(int(rng.integers(0, 300000)))
    yield (rng.integers(0, 256, 150000, dtype=np.uint8) & rng.integers(0, 256, 150000, dtype=np.uint8)).tobytes()
    yield rng.integers(0, 4096, 100000, dtype=np.uint16).tobytes()
    yield (bytes(rng.integers(0, 256, 37, dtype=np.uint8)) * 5000)[: int(rng.integers(1, 180000))]
    yield bytes(rng.integers(0, 4, int(rng.integers(0, 64)), dtype=np.uint8))


def test_random_frames_at_many_levels(zd):
    rng = np.random.default_rng(5)
    z = F.zstd()
    ok = total = 0
    for _ in range(3):
        for data in _samples(rng):
            for lvl in (-3, 1, 3, 6, 12, 19):
                fr = z.compress(data, lvl)
                rc, got = zd(fr)
                assert rc in (0, 1) and (rc == 1 or got == data), (len(data), lvl)
                if len(data) > zd.max_content:
                    assert rc == 1
                    continue
                ok += rc == 0
                total += 1
    payload = b"\x07" * 97 + np.stack([rng.integers(0, 1 << 36, 4096, dtype=np.uint64) for _ in range(4)]).tobytes()
    assert ok >= total - 6, "only frames beyond the decoder's limits (blocks, sequences) may be handed back"
    rc, got = zd(F.zstd_structured_frame(payload))
    assert rc == 0 and got == payload


def test_mutated_frames_never_decode_wrongly(zd):
    rng = np.random.default_rng(6)
    z = F.zstd()
    base = [z.compress(d, 3) for d in _samples(rng)] + [z.compress(d, 19) for d in _samples(rng)]
    accepted = handed_back = 0
    for it in range(1500):
        fr = bytearray(base[it % len(base)])
        if not fr:
            continue
        kind = it % 4
        if kind == 0:
            fr = fr[: rng.integers(0, len(fr))]
        elif kind == 1:
            for _ in range(rng.integers(1, 4)):
                fr[rng.integers(0, len(fr))] ^= 1 << rng.integers(0, 8)
        elif kind == 2:
            fr += bytes(rng.integers(0, 256, rng.integers(1, 9), dtype=np.uint8))
        else:
            i = rng.integers(0, len(fr))
            fr[i : i + 4] = bytes(rng.integers(0, 256, 4, dtype=np.uint8))
        fr = bytes(fr)
        rc, got = zd(fr)
        if rc == 0:
            want = _reference(fr)
            assert want is not None and got == want, "decoded something libzstd rejects or decodes differently"
            accepted += 1
        else:
            handed_back += 1
    assert accepted > 100 and handed_back > 100


def test_parallel_executor_resolves_ciphertext_frames_by_jumping(zd):
    """zstd_exec3.h on what it is built for: a level-3 ciphertext frame has ~16 k matches in 16 dependency chains ~1,000 long
    (the top-nibble tails), most 5-byte matches read a literal followed by a match.  The pointer jumping (with the one split)
    must leave next to nothing to the copy phase's polling, in a logarithmic number of rounds."""
    rng = np.random.default_rng(8)
    q = (0xFFFFEE001, 0xFFFFC4001)
    z = F.zstd()
    for _ in range(4):
        data = bytes(rng.integers(0, 256, 97, dtype=np.uint8)) + np.stack(
            [rng.integers(0, q[l], 4096, dtype=np.uint64) for _ in range(2) for l in range(2)]).tobytes()
        for lvl in (1, 3, 7):
            rc, got = zd(z.compress(data, lvl))
            assert rc == 0 and got == data
            assert zd.rounds <= 24 and zd.polls <= 2000, (lvl, zd.rounds, zd.polls)
    rc, got = zd(F.zstd_structured_frame(data))  # one chain of 16,382 matches at offset 8
    assert rc == 0 and got == data and zd.rounds <= 24
