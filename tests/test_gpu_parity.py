"""GPU parity: every kernel behind the C ABI, bit-compared with the CPU oracle on the same inputs.
Bar: bit-exact (integer work).  Run on the B200 box: pytest -m gpu."""
import os

import numpy as np
import pytest

from helpers import KINDS, MODULI, N, ROOT, REF_A, REF_B, REF_EXPECT, decrypt_value, encrypt_value, oracle_binary, plain_u16, precompile_name, random_ct, value_of
from oracle import bfv
from oracle import formats as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["seal", "structured"], autouse=True)
def writer_mode(request):
    """every test of this file runs under both result writers: "seal" (default: libzstd level 3, the bytes SEAL's save() writes)
    and "structured" (fhe_b200_set_zstd_writer(1): frames laid out directly, written on the GPU in tiles / single calls)."""
    from fhe_precompiles_b200 import _lib

    L = _lib.lib()
    prev = L.fhe_b200_set_zstd_writer(1 if request.param == "structured" else 0)
    yield request.param
    L.fhe_b200_set_zstd_writer(prev)


def STRUCT() -> bool:
    """is the structured writer active? (expected result bytes follow the library's current writer)"""
    from fhe_precompiles_b200 import _lib

    return bool(_lib.lib().fhe_b200_set_zstd_writer(-1))


@pytest.fixture(scope="module")
def dev():
    import torch

    from fhe_precompiles_b200 import device

    assert torch.cuda.is_available(), "no CUDA device: the product has no CPU path"
    device.init(0)
    return device


def to_dev(a: np.ndarray):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()


def to_np(t) -> np.ndarray:
    return t.cpu().numpy().view(np.uint64)


def edge_ct(n_rand: int, seed: int) -> np.ndarray:
    """random residues plus the edge polynomials: all zero, all q-1, single max coefficient"""
    rng = np.random.default_rng(seed)
    cts = random_ct(rng, n_rand + 3)
    cts[n_rand] = 0
    for l in range(2):
        cts[n_rand + 1, :, l, :] = MODULI[l] - 1
    cts[n_rand + 2] = 0
    cts[n_rand + 2, 0, 0, 0] = MODULI[0] - 1
    cts[n_rand + 2, 1, 1, N - 1] = MODULI[1] - 1
    return cts


@pytest.mark.parametrize("mod", range(6))
def test_ntt_forward_inverse(dev, mod):
    rng = np.random.default_rng(100 + mod)
    x = rng.integers(0, MODULI[mod], size=(5, N), dtype=np.uint64)
    x[3] = 0
    x[4] = MODULI[mod] - 1
    want = bfv.ntt_fwd(x, mod)
    d = to_dev(x)
    dev.ntt_(d, [mod], inverse=False)
    got = to_np(d)
    assert np.array_equal(got, want)
    dev.ntt_(d, [mod], inverse=True)
    assert np.array_equal(to_np(d), x)
    # inverse on arbitrary canonical input too
    y = to_dev(x)
    dev.ntt_(y, [mod], inverse=True)
    assert np.array_equal(to_np(y), bfv.ntt_inv(x, mod))


def test_ntt_mixed_limbs(dev):
    rng = np.random.default_rng(7)
    x = np.stack([rng.integers(0, MODULI[m], size=(4, N), dtype=np.uint64) for m in (0, 1, 2)], axis=1)  # [4][3][N]
    d = to_dev(x)
    dev.ntt_(d, [0, 1, 2])
    got = to_np(d)
    for m in range(3):
        assert np.array_equal(got[:, m], bfv.ntt_fwd(x[:, m], m))


def test_add_sub_negate(dev):
    a, b = edge_ct(5, 1), edge_ct(5, 2)[::-1].copy()
    da, db = to_dev(a), to_dev(b)
    assert np.array_equal(to_np(dev.add(da, db)), np.stack([bfv.add(x, y) for x, y in zip(a, b)]))
    assert np.array_equal(to_np(dev.sub(da, db)), np.stack([bfv.sub(x, y) for x, y in zip(a, b)]))
    assert np.array_equal(to_np(dev.negate(da)), np.stack([bfv.negate(x) for x in a]))


def test_plain_ops(dev):
    import torch

    cts = edge_ct(5, 3)
    rng = np.random.default_rng(4)
    plains = rng.integers(0, 4096, size=(len(cts), N), dtype=np.uint16)
    plains[0] = 0
    plains[1] = 4095
    plains[2] = 0
    plains[2, 5] = 2048  # exactly the upper-half threshold
    dct = to_dev(cts)
    dpl = torch.from_numpy(plains.view(np.int16)).cuda()
    for mode, fn in ((0, bfv.add_plain), (1, bfv.sub_plain), (3, lambda c, p: bfv.negate(bfv.sub_plain(c, p)))):
        got = to_np(dev.plain_addsub(dct, dpl, mode))
        want = np.stack([fn(c, p.astype(np.uint64)) for c, p in zip(cts, plains)])
        assert np.array_equal(got, want), f"plain_addsub mode {mode}"
    got = to_np(dev.multiply_plain(dct, dpl))
    want = np.stack([bfv.multiply_plain(c, p.astype(np.uint64)) for c, p in zip(cts, plains)])
    assert np.array_equal(got, want)


def test_multiply_against_oracle_behz_stages(dev):
    """multiply on edge inputs against the oracle's BEHZ stages: fastbconv_m_tilde + sm_mrq, NTT + tensor + INTT * t,
    fast_floor + fastbconv_sk"""
    a, b = edge_ct(3, 5), edge_ct(3, 6)[::-1].copy()
    want_c3 = np.stack([bfv.behz_floor_sk(bfv.behz_tensor(bfv.behz_extend(x, y))) for x, y in zip(a, b)])
    assert np.array_equal(to_np(dev.multiply(to_dev(a), to_dev(b))), want_c3), "bfv_multiply"


def test_relinearize_and_mul_relin(dev, keys):
    a, b = edge_ct(3, 8), edge_ct(3, 9)[::-1].copy()
    da, db, drk = to_dev(a), to_dev(b), to_dev(keys.rk)
    c3 = np.stack([bfv.multiply(x, y) for x, y in zip(a, b)])
    want = np.stack([bfv.relinearize(c, keys.rk) for c in c3])
    assert np.array_equal(to_np(dev.relinearize(to_dev(c3), drk)), want), "switch_key_inplace"
    assert np.array_equal(to_np(dev.mul_relin(da, db, drk)), want), "multiply + relinearize"


def test_mul_relin_real_encryptions_chunked(dev, keys):
    """batch larger than the engine's chunk (set to 128 ops here: chunks of 128, 128 and 44): bit-exact vs the oracle on a
    sample that straddles every chunk boundary, all decrypt."""
    rng = np.random.default_rng(2)
    n = 300
    vals_a = rng.integers(-(2**15), 2**15, size=n)
    vals_b = rng.integers(-(2**15), 2**15, size=n)
    a = np.stack([encrypt_value(keys, "i64", int(v), 1000 + i) for i, v in enumerate(vals_a)])
    b = np.stack([encrypt_value(keys, "i64", int(v), 5000 + i) for i, v in enumerate(vals_b)])
    prev = dev.set_chunk_ops(128)
    try:
        assert dev.set_chunk_ops(0) == 128
        out = to_np(dev.mul_relin(to_dev(a), to_dev(b), to_dev(keys.rk)))
        c3 = to_np(dev.multiply(to_dev(a), to_dev(b)))
        out2 = to_np(dev.relinearize(to_dev(c3), to_dev(keys.rk)))
    finally:
        dev.set_chunk_ops(prev)
    assert np.array_equal(out, out2), "multiply then relinearize, chunked, equals the fused call"
    for i in list(range(0, n, 37)) + [127, 128, 129, 255, 256, 257, n - 1]:
        assert np.array_equal(out[i], bfv.mul_relin(a[i], b[i], keys.rk)), f"op {i}"
    for i in range(0, n, 5):
        assert decrypt_value(keys, "i64", out[i]) == int(vals_a[i]) * int(vals_b[i])
    # one chunk (the default 4,096) gives the same bits
    assert np.array_equal(to_np(dev.mul_relin(to_dev(a), to_dev(b), to_dev(keys.rk))), out)


def test_mul_relin_more_than_one_default_chunk(dev, keys):
    """n > 4,096 at the default chunk size (what config 4's 65,536 calls need): Engine::mul_relin's second chunk.  Ops are
    drawn from a pool of 67 distinct random ciphertexts so the expected values cost 67 oracle calls."""
    import torch

    assert dev.set_chunk_ops(0) == 4096
    n, pool = 4096 + 203, 67
    rng = np.random.default_rng(77)
    pa, pb = random_ct(rng, pool), random_ct(rng, pool)
    idx = torch.arange(n) % pool
    a, b = to_dev(pa)[idx.cuda()].contiguous(), to_dev(pb)[idx.cuda()].contiguous()
    out = dev.mul_relin(a, b, to_dev(keys.rk))
    want = to_dev(np.stack([bfv.mul_relin(pa[i], pb[i], keys.rk) for i in range(pool)]))
    assert torch.equal(out, want[idx.cuda()]), "every op of both chunks"


def test_streams_do_not_share_scratch(dev, keys):
    """two streams on one GPU, interleaved enqueues from one thread and concurrent enqueues from two threads: each
    (device, stream) has its own scratch arena, so results are bit-exact (they used to overwrite each other's scratch)."""
    import threading

    import torch

    rng = np.random.default_rng(31)
    n = 96
    a, b = random_ct(rng, n), random_ct(rng, n)
    rk = to_dev(keys.rk)
    want = dev.mul_relin(to_dev(a), to_dev(b), rk)
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    da, db = to_dev(a), to_dev(b)
    outs = []
    for rep in range(6):
        for s in (s1, s2):
            with torch.cuda.stream(s):
                outs.append(dev.mul_relin(da, db, rk))
    torch.cuda.synchronize()
    assert all(torch.equal(o, want) for o in outs)

    res = {}

    def worker(k):
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            mine = [dev.mul_relin(da, db, rk) for _ in range(8)]
        s.synchronize()
        res[k] = all(torch.equal(o, want) for o in mine)

    ts = [threading.Thread(target=worker, args=(k,)) for k in range(6)]  # more threads than idle arenas kept per device
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert res == {k: True for k in range(6)}


# ---------------------------------------------------------------- the byte surface (C ABI part 1)
SHAPES = ("ctct", "ctpt", "ptct")


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("op", ("add", "sub", "mul"))
@pytest.mark.parametrize("shape", SHAPES)
def test_precompile_matches_reference_tests(keys, kind, op, shape):
    """fhe.rs:1070-2076 `precompile_*_works`: 16 op 4 through pack_binary_operation -> precompile ->
    deserialize -> decrypt; plus byte equality with the oracle's result serialised by the format oracle."""
    from fhe_precompiles_b200 import FHE, pack

    a_val, b_val = value_of(kind, REF_A), value_of(kind, REF_B)
    ct_a = encrypt_value(keys, kind, a_val, 11)
    ct_b = encrypt_value(keys, kind, b_val, 12)
    ser = lambda ct: F.make_ciphertext(kind, ct).to_bytes()
    if shape == "ctct":
        args, oargs = (ser(ct_a), ser(ct_b)), (ct_a, ct_b)
    elif shape == "ctpt":
        args, oargs = (ser(ct_a), pack.SERIALIZE[kind](b_val)), (ct_a, b_val)
    else:
        args, oargs = (pack.SERIALIZE[kind](a_val), ser(ct_b)), (a_val, ct_b)
    name = precompile_name(op, shape, kind)
    out = getattr(FHE, name)(pack.pack_binary_operation(keys.pub_bytes, *args))
    want = oracle_binary(op, shape, kind, *oargs, keys.rk)
    assert out == F.make_ciphertext(kind, want).to_bytes(structured=STRUCT()), "packed ciphertext bytes differ from the oracle's"
    got_ct = F.Ciphertext.from_bytes(out)
    assert decrypt_value(keys, kind, got_ct.polys()) == value_of(kind, REF_EXPECT[op])


def test_precompile_errors(keys):
    from fhe_precompiles_b200 import FHE, FheError, pack

    ct = F.make_ciphertext("i64", encrypt_value(keys, "i64", 3, 1)).to_bytes()
    good = pack.pack_binary_operation(keys.pub_bytes, ct, ct)

    def code(fn, data):
        with pytest.raises(FheError) as e:
            fn(data)
        return e.value.code

    assert code(FHE.add_cipheri64_cipheri64, b"\x00\x01") == 1  # pack.rs:244-246
    assert code(FHE.add_cipheri64_cipheri64, good[:8] + b"junk" + good[12:]) == 3  # key fails to deserialize
    assert code(FHE.add_cipheri64_i64, pack.pack_binary_operation(keys.pub_bytes, ct, b"\x00" * 7)) == 3  # pack.rs:86
    assert code(FHE.add_cipheru64_cipheru64, good) == 7  # argument type mismatch -> sunscreen runtime error
    bad_off = bytearray(good)
    bad_off[0:4] = (len(good) + 5).to_bytes(4, "big")
    assert code(FHE.add_cipheri64_cipheri64, bytes(bad_off)) == 1  # reference panics; we bounds-check
    # transparent result must be accepted (fhe.rs:2124-2140): ct - ct = all-zero ciphertext
    out = FHE.sub_cipheri64_cipheri64(good)
    assert not F.Ciphertext.from_bytes(out).polys().any()


def test_batch_surface(keys):
    from fhe_precompiles_b200 import FHE, pack

    calls, wants = [], []
    for i in range(12):
        kind = KINDS[i % 4]
        a, b = encrypt_value(keys, kind, value_of(kind, 3 + i), 50 + i), encrypt_value(keys, kind, value_of(kind, 2), 90 + i)
        sa, sb = (F.make_ciphertext(kind, x).to_bytes() for x in (a, b))
        op = ("add", "sub", "mul")[i % 3]
        calls.append((precompile_name(op, "ctct", kind), pack.pack_binary_operation(keys.pub_bytes, sa, sb)))
        wants.append(F.make_ciphertext(kind, oracle_binary(op, "ctct", kind, a, b, keys.rk)).to_bytes(structured=STRUCT()))
    calls.append(("add_cipheri64_cipheri64", b"\x00"))
    res = FHE.run_batch(calls, host_threads=4)
    assert [r[0] for r in res[:-1]] == [0] * 12 and res[-1][0] == 1
    for (st, out), want in zip(res[:-1], wants):
        assert out == want


def test_batch_tiles_equal_single_calls(keys):
    """fhe_b200_batch runs tiles of calls through one lane (Engine::binary_tile): every operation class, two keys, and an error
    at each stage of the reference's decode order must give exactly the status and bytes of the single-call symbol."""
    from fhe_precompiles_b200 import FHE, FheError, pack

    rng = np.random.default_rng(404)
    pk_no_relin = F.PublicKey(F.PublicKey.from_bytes(keys.pub_bytes).public_key, None, None).to_bytes()
    calls = []
    for i in range(44):
        kind = KINDS[i % 4]
        op = ("add", "sub", "mul")[(i // 4) % 3]
        shape = SHAPES[(i // 2) % 3]
        va, vb = value_of(kind, 2 + i % 5), value_of(kind, 1 + i % 3)
        ca = F.make_ciphertext(kind, encrypt_value(keys, kind, va, 500 + i)).to_bytes()
        cb = F.make_ciphertext(kind, encrypt_value(keys, kind, vb, 600 + i)).to_bytes(structured=bool(i & 1))
        sc = pack.SERIALIZE[kind](vb)
        args = {"ctct": (ca, cb), "ctpt": (ca, sc), "ptct": (sc, cb)}[shape]
        pkb = keys.net_pub_bytes if i % 7 == 3 else keys.pub_bytes
        data = pack.pack_binary_operation(pkb, *args)
        fault = i % 11
        if fault == 4:
            data = data[:9]  # framing: code 1
        elif fault == 5:
            data = pack.pack_binary_operation(pkb[:-5], *args)  # key does not deserialise: 3
        elif fault == 6 and shape != "ptct":
            data = pack.pack_binary_operation(pkb, ca[:-7], args[1])  # operand a: 3
        elif fault == 7 and shape == "ctct":
            other = KINDS[(i + 1) % 4]
            data = pack.pack_binary_operation(pkb, ca, F.make_ciphertext(other, encrypt_value(keys, other, 1, 9)).to_bytes())  # type: 7
        elif fault == 8:
            data = pack.pack_binary_operation(pk_no_relin, *args)  # missing relin keys: 7 for ct*ct only
        calls.append((precompile_name(op, shape, kind), data))
    want = []
    for name, data in calls:
        try:
            want.append((0, getattr(FHE, name)(data)))
        except FheError as e:
            want.append((e.code, b""))
    assert {st for st, _ in want} >= {0, 1, 3, 7}
    for threads in (1, 2, 16):
        got = FHE.run_batch(calls, host_threads=threads)
        assert [g[0] for g in got] == [w[0] for w in want], threads
        assert all(g[1] == w[1] for g, w in zip(got, want)), threads
    order = rng.permutation(len(calls))
    got = FHE.run_batch([calls[i] for i in order], host_threads=2)
    assert all(got[k] == want[i] for k, i in enumerate(order))


def test_device_zstd_inflate_matches_libzstd(dev):
    """The device zstd decoder (k_zd2_parse, k_zd3_huf, k_zd3_seq, k_zd3_exec): ciphertext-payload frames written by libzstd
    at several levels, by the structured writer, other content of the same size (Huffman literals, RLE, raw blocks) and
    corrupted frames. A frame the device accepts must be byte-identical to libzstd's output; everything else must be handed
    back (status 2)."""
    import ctypes

    from fhe_precompiles_b200 import _lib

    L = _lib.lib()
    z = F.zstd()
    rng = np.random.default_rng(2024)
    size = 97 + 8 * 4 * N
    ct = lambda: bytes(rng.integers(0, 256, 97, dtype=np.uint8)) + np.stack(
        [rng.integers(0, MODULI[l], N, dtype=np.uint64) for _ in range(2) for l in range(2)]).tobytes()
    text = bytes(rng.choice(list(b"abcdefgh \n"), size=size).astype(np.uint8))
    payloads = [ct() for _ in range(6)] + [text, bytes(size), rng.integers(0, 256, size, dtype=np.uint8).tobytes()]
    levels = [-3, 1, 3, 7, 12, 19, 3, 3, 3]
    frames = [z.compress(p, lvl) for p, lvl in zip(payloads, levels)]
    payloads.append(payloads[0]), frames.append(F.zstd_structured_frame(payloads[0]))
    good = len(frames)
    for it in range(40):  # corrupted variants
        fr = bytearray(frames[it % 6])
        if it % 3 == 0:
            fr[rng.integers(0, len(fr))] ^= 1 << rng.integers(0, 8)
        elif it % 3 == 1:
            fr = fr[: rng.integers(1, len(fr))]
        else:
            i = rng.integers(0, len(fr) - 4)
            fr[i : i + 4] = bytes(rng.integers(0, 256, 4, dtype=np.uint8))
        frames.append(bytes(fr))
        try:
            ok = z.lib.ZSTD_getFrameContentSize(frames[-1], len(frames[-1])) == size
            payloads.append(z.decompress(frames[-1]) if ok else None)
        except ValueError:
            payloads.append(None)
    n = len(frames)
    bufs = [ctypes.create_string_buffer(f, len(f)) for f in frames]
    ptrs = (ctypes.c_void_p * n)(*[ctypes.cast(b, ctypes.c_void_p) for b in bufs])
    lens = (ctypes.c_size_t * n)(*[len(f) for f in frames])
    out = ctypes.create_string_buffer(n * size)
    status = (ctypes.c_int32 * n)()
    ms = ctypes.c_float()
    assert L.fhe_b200_zstd_inflate(0, ptrs, lens, n, out, status, ctypes.byref(ms)) == 0
    raw = out.raw
    assert list(status[:good]) == [1] * good, "every well-formed frame is inflated on the device"
    for i in range(n):
        assert status[i] in (1, 2)
        if status[i] == 1:
            assert payloads[i] is not None and raw[i * size : (i + 1) * size] == payloads[i], i


@pytest.mark.parametrize("host_pct,writer", [("0", "0"), ("40", "0"), ("40", "1")])
def test_batch_tiles_with_device_zstd(keys, host_pct, writer):
    """FHE_B200_DEVICE_ZSTD=1: the operands of a tile are inflated by the device decoder (k_zd2_parse / k_zd3_seq / k_zd3_exec)
    instead of libzstd - all of them, or (FHE_B200_HOST_INFLATE_PCT=40) a hybrid tile whose device share is decoded while the
    host inflates the rest.  Same statuses and bytes as the single-call symbols, with either result writer (the knobs are read
    when the engine starts, hence the subprocess)."""
    import subprocess
    import sys

    code = """
import sys
sys.path.insert(0, %r); sys.path.insert(0, %r)
import numpy as np
from helpers import KeySet, KINDS, encrypt_value, precompile_name, value_of
from fhe_precompiles_b200 import FHE, FheError, pack
from oracle import formats as F
keys = KeySet.load()
calls = []
for i in range(24):
    kind = KINDS[i %% 4]; op = ("add", "sub", "mul")[(i // 4) %% 3]; shape = ("ctct", "ctpt", "ptct")[(i // 2) %% 3]
    va, vb = value_of(kind, 2 + i %% 5), value_of(kind, 1 + i %% 3)
    ca = F.make_ciphertext(kind, encrypt_value(keys, kind, va, 700 + i)).to_bytes()
    cb = F.make_ciphertext(kind, encrypt_value(keys, kind, vb, 800 + i)).to_bytes(structured=bool(i & 1))
    sc = pack.SERIALIZE[kind](vb)
    args = {"ctct": (ca, cb), "ctpt": (ca, sc), "ptct": (sc, cb)}[shape]
    data = pack.pack_binary_operation(keys.pub_bytes, *args)
    if i %% 9 == 4: data = pack.pack_binary_operation(keys.pub_bytes, ca[:-9], args[1]) if shape != "ptct" else data[:11]
    if i %% 9 == 7:
        bad = bytearray(ca); bad[-300] ^= 0x10
        data = pack.pack_binary_operation(keys.pub_bytes, bytes(bad), args[1]) if shape != "ptct" else data
    calls.append((precompile_name(op, shape, kind), data))
want = []
for name, data in calls:
    try: want.append((0, getattr(FHE, name)(data)))
    except FheError as e: want.append((e.code, b""))
got = FHE.run_batch(calls, host_threads=2)
assert got == want, [(g[0], w[0]) for g, w in zip(got, want)]
assert sum(1 for st, _ in want if st == 0) >= 16 and any(st for st, _ in want)
print("device-zstd tiles ok")
""" % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ, FHE_B200_DEVICE_ZSTD="1", FHE_B200_HOST_INFLATE_PCT=host_pct, FHE_B200_ZSTD_WRITER=writer)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "device-zstd tiles ok" in r.stdout, r.stdout + r.stderr


def test_writer_modes_and_chained_calls(keys):
    """default / fhe_b200_set_zstd_writer(0): outputs are libzstd level-3 frames, byte-identical to the format oracle's default
    serialisation (what SEAL's save() writes; pinned by the reference's known answers).  fhe_b200_set_zstd_writer(1): structured
    frames.  Outputs of one call are valid inputs of the next in either mode."""
    from fhe_precompiles_b200 import FHE, _lib, pack

    a, b = encrypt_value(keys, "i64", 6, 401), encrypt_value(keys, "i64", -7, 402)
    sa, sb = (F.make_ciphertext("i64", x).to_bytes() for x in (a, b))
    packed = pack.pack_binary_operation(keys.pub_bytes, sa, sb)
    prod = bfv.mul_relin(a, b, keys.rk)
    L = _lib.lib()
    prev = L.fhe_b200_set_zstd_writer(-1)
    try:
        for mode in (0, 1):
            L.fhe_b200_set_zstd_writer(mode)
            out1 = FHE.mul_cipheri64_cipheri64(packed)
            assert out1 == F.make_ciphertext("i64", prod).to_bytes(structured=bool(mode))
            out2 = FHE.add_cipheri64_cipheri64(pack.pack_binary_operation(keys.pub_bytes, out1, sa))  # a result as input
            assert out2 == F.make_ciphertext("i64", bfv.add(prod, a)).to_bytes(structured=bool(mode))
    finally:
        L.fhe_b200_set_zstd_writer(prev)
    assert decrypt_value(keys, "i64", F.Ciphertext.from_bytes(out2).polys()) == -42 + 6


# ---------------------------------------------------------------- encrypt / decrypt (config 5, threshold API)
def test_device_decrypt_matches_oracle(dev, keys):
    import torch

    rng = np.random.default_rng(21)
    vals = [int(v) for v in rng.integers(-(2**40), 2**40, size=24)]
    cts = np.stack([encrypt_value(keys, "i64", v, 300 + i) for i, v in enumerate(vals)])
    prod = np.stack([bfv.mul_relin(cts[i], cts[(i + 1) % len(cts)], keys.rk) for i in range(4)])  # noisier inputs too
    allct = np.concatenate([cts, prod])
    plain = dev.decrypt(to_dev(allct), to_dev(keys.sk)).cpu().numpy().view(np.uint16)
    for i, ct in enumerate(allct):
        want, budget = bfv.decrypt(ct, keys.sk)
        assert budget > 0
        assert np.array_equal(plain[i].astype(np.uint64), want), f"ciphertext {i}"
    assert [bfv.decode("i64", p.astype(np.uint64)) for p in plain[: len(vals)]] == vals


def test_device_encrypt_roundtrip(dev, keys):
    """config 5 shape: pk-encrypt random i64 under the network key on the GPU, decrypt with network.pri, all equal;
    the GPU sampler is the library's own, so the check is decrypt-equality, noise budget and determinism."""
    import torch

    rng = np.random.default_rng(5)
    n = 64
    vals = [int(v) for v in rng.integers(-(2**62), 2**62, size=n)]
    plains = np.stack([plain_u16("i64", v) for v in vals])
    seeds = torch.arange(1000 * 8, (1000 + n) * 8, dtype=torch.int64).reshape(n, 8).cuda()
    dpl = torch.from_numpy(plains.view(np.int16)).cuda()
    dpk = to_dev(keys.net_pk)
    ct = dev.encrypt(dpk, dpl, seeds)
    ct2 = dev.encrypt(dpk, dpl, seeds)
    assert torch.equal(ct, ct2), "deterministic in (seed, plaintext, key)"
    cts = to_np(ct)
    assert not np.array_equal(cts[0, 1], cts[1, 1]), "different seeds give different randomness"
    for l in range(2):
        assert (cts[:, :, l, :] < MODULI[l]).all()
    for i in range(n):
        plain, budget = bfv.decrypt(cts[i], keys.net_sk)
        assert 47 <= budget <= 51, f"fresh noise budget {budget}"
        assert bfv.decode("i64", plain) == vals[i]
    # the deterministic encrypt works at the data level (no modulus switching): 49 bits of budget, 4 below stock SEAL's 53
    assert np.median([bfv.decrypt(c, keys.net_sk)[1] for c in cts[:16]]) == 49
    # GPU decrypt agrees
    got = dev.decrypt(ct, to_dev(keys.net_sk)).cpu().numpy().view(np.uint16)
    assert np.array_equal(got[:, :64], plains[:, :64]) and not got[:, 64:].any()
    # and the ciphertexts multiply correctly under the network relin keys
    prod = to_np(dev.mul_relin(ct[:8], ct[8:16], to_dev(keys.net_rk)))
    for i in range(8):
        assert bfv.decode("i64", bfv.decrypt(prod[i], keys.net_sk)[0]) == (vals[i] * vals[8 + i] + 2**63) % 2**64 - 2**63


@pytest.mark.parametrize("kind,value", [("u256", 12), ("u64", 12), ("i64", 12), ("frac64", 12.0), ("i64", -7), ("frac64", -2.75),
                                        ("u256", 2**200 + 5), ("u64", 2**64 - 1)])
def test_threshold_api_roundtrip(keys, kind, value):
    """fhe.rs:2248-2303 fhe_decrypt_test: encrypt -> decrypt round trip for all four types (value 12), plus edge values."""
    from fhe_precompiles_b200 import FHE, pack

    ser = pack.SERIALIZE[kind](value)
    enc = getattr(FHE, f"encrypt_{kind}")(pack.pack_two_arguments(ser, bytes([1, 2, 3])))
    assert getattr(FHE, f"encrypt_{kind}")(pack.pack_two_arguments(ser, bytes([1, 2, 3]))) == enc  # deterministic
    assert getattr(FHE, f"encrypt_{kind}")(pack.pack_two_arguments(ser, bytes([1, 2, 4]))) != enc  # seed depends on public data
    ct = F.Ciphertext.from_bytes(enc)
    assert decrypt_value(keys, kind, ct.polys(), network=True) == value_of(kind, value)
    dec = getattr(FHE, f"decrypt_{kind}")(pack.pack_one_argument(enc))
    assert pack.deserialize_scalar(kind, dec) == value_of(kind, value)


def test_encrypt_same_seed_and_value_works(keys):
    """fhe.rs:2124-2140: two identical encrypts subtract to a transparent ciphertext that decrypts to 0."""
    from fhe_precompiles_b200 import FHE, pack

    inp = pack.pack_two_arguments(pack.serialize_u256(16), bytes([1, 2, 3, 4]))
    a, b = FHE.encrypt_u256(inp), FHE.encrypt_u256(inp)
    out = FHE.sub_cipheru256_cipheru256(pack.pack_binary_operation(keys.net_pub_bytes, a, b))
    assert pack.deserialize_scalar("u256", FHE.decrypt_u256(out)) == 0


def test_reencrypt(keys):
    """fhe.rs:2143-2245 fhe_refresh_test / fhe_reencrypt_test without the SEAL-PRNG-dependent SHA-512 KATs:
    encrypt under the network key, reencrypt to tests/data/public_key.bin, decrypt with tests/data/private_key.bin."""
    from fhe_precompiles_b200 import FHE, FheError, pack

    enc = FHE.encrypt_u256(pack.pack_two_arguments(pack.serialize_u256(12), bytes([1, 2, 3])))
    re = FHE.reencrypt_u256(pack.pack_binary_operation(keys.pub_bytes, enc, bytes([1, 2, 3])))
    assert decrypt_value(keys, "u256", F.Ciphertext.from_bytes(re).polys()) == 12
    re_net = FHE.reencrypt_u256(pack.pack_binary_operation(keys.net_pub_bytes, enc, bytes([1, 2, 3])))
    assert pack.deserialize_scalar("u256", FHE.decrypt_u256(re_net)) == 12
    assert FHE.public_key_bytes() == keys.net_pub_bytes
    with pytest.raises(FheError) as e:
        FHE.decrypt_i64(enc)  # a u256 ciphertext is not an i64 ciphertext
    assert e.value.code == 5


# ---------------------------------------------------------------- full-size, size-independent properties
def test_full_batch_roundtrip_properties(dev, keys):
    """BASELINE config 3 size (4,096 ops): encrypt -> multiply+relinearise -> decrypt equals the plaintext products for every
    op; (a + b) - b == a and a - a == 0 bit-exactly; 64 ops spot-checked bit-exactly against the oracle."""
    import torch

    n = 4096
    rng = np.random.default_rng(2)
    va = rng.integers(-(2**15), 2**15, n)
    vb = rng.integers(-(2**15), 2**15, n)

    def plains(vals):
        mag = np.abs(vals).astype(np.uint64)
        bits = ((mag[:, None] >> np.arange(64, dtype=np.uint64)[None, :]) & 1).astype(np.int64)
        out = np.zeros((len(vals), N), dtype=np.int16)
        out[:, :64] = np.where(vals[:, None] < 0, bits * 4095, bits).astype(np.uint16).view(np.int16)
        return torch.from_numpy(out).cuda()

    pk, rk, sk = to_dev(keys.net_pk), to_dev(keys.net_rk), to_dev(keys.net_sk)
    a = dev.encrypt(pk, plains(va), torch.arange(8 * n, dtype=torch.int64).reshape(n, 8).cuda())
    b = dev.encrypt(pk, plains(vb), torch.arange(8 * n, 16 * n, dtype=torch.int64).reshape(n, 8).cuda())
    prod = dev.mul_relin(a, b, rk)
    dec = dev.decrypt(prod, sk).cpu().numpy().view(np.uint16).astype(np.int64)
    dec = np.where(dec >= 2048, dec - 4096, dec)  # centred coefficients; value = sum c_i 2^i
    got = (dec[:, :64] * (1 << np.arange(64, dtype=np.int64))[None, :]).sum(axis=1)  # products < 2^31: no wrap
    assert np.array_equal(got, va * vb)
    s = dev.add(a, b)
    assert torch.equal(dev.sub(s, b), a)
    assert not dev.sub(a, a).any()
    assert torch.equal(dev.negate(dev.negate(a)), a)
    an, bn, pn = to_np(a), to_np(b), to_np(prod)
    for i in range(0, n, 64):
        assert np.array_equal(pn[i], bfv.mul_relin(an[i], bn[i], keys.net_rk)), f"op {i}"


def test_empty_batches(dev, keys):
    import torch

    e = torch.empty((0, 2, 2, N), dtype=torch.int64, device="cuda")
    rk = to_dev(keys.rk)
    assert dev.add(e, e).shape[0] == 0 and dev.mul_relin(e, e, rk).shape[0] == 0 and dev.multiply(e, e).shape[0] == 0
    from fhe_precompiles_b200 import FHE

    assert FHE.run_batch([]) == []


# ---------------------------------------------------------------- re-entrancy and the key cache
def test_concurrent_calls_and_key_cache_eviction(keys, monkeypatch):
    """the C ABI is re-entrant like the reference's global FheApp (testnet.rs:25): 8 threads x mixed precompiles under
    4 distinct public keys with a 2-entry key cache (forcing evictions while other threads hold keys); every result must
    equal the oracle's bytes."""
    import threading

    from fhe_precompiles_b200 import FHE, pack

    monkeypatch.setenv("FHE_B200_KEY_CACHE", "2")
    t_pk, n_pk = F.PublicKey.from_bytes(keys.pub_bytes), F.PublicKey.from_bytes(keys.net_pub_bytes)
    variants = [
        (keys.pub_bytes, keys.rk),
        (keys.net_pub_bytes, keys.net_rk),
        (F.PublicKey(t_pk.public_key, None, n_pk.relin_key).to_bytes(), keys.net_rk),
        (F.PublicKey(n_pk.public_key, None, t_pk.relin_key).to_bytes(), keys.rk),
    ]
    a, b = encrypt_value(keys, "i64", 21, 70), encrypt_value(keys, "i64", -3, 71)
    sa, sb = (F.make_ciphertext("i64", x).to_bytes() for x in (a, b))
    want = {}
    for vi, (pkb, rk) in enumerate(variants):
        want[("mul", vi)] = F.make_ciphertext("i64", bfv.mul_relin(a, b, rk)).to_bytes(structured=STRUCT())
        want[("add", vi)] = F.make_ciphertext("i64", bfv.add(a, b)).to_bytes(structured=STRUCT())
        want[("mulp", vi)] = F.make_ciphertext("i64", bfv.multiply_plain(a, bfv.encode("i64", 5))).to_bytes(structured=STRUCT())
    errors = []

    def worker(tid):
        try:
            for it in range(6):
                vi = (tid + it) % 4
                pkb = variants[vi][0]
                kind = ("mul", "add", "mulp")[(tid + it) % 3]
                if kind == "mul":
                    out = FHE.mul_cipheri64_cipheri64(pack.pack_binary_operation(pkb, sa, sb))
                elif kind == "add":
                    out = FHE.add_cipheri64_cipheri64(pack.pack_binary_operation(pkb, sa, sb))
                else:
                    out = FHE.mul_cipheri64_i64(pack.pack_binary_operation(pkb, sa, pack.serialize_i64(5)))
                if out != want[(kind, vi)]:
                    errors.append((tid, it, kind, vi))
        except Exception as e:  # noqa: BLE001
            errors.append((tid, repr(e)))

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(8)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


def test_plain_c_caller(keys, tmp_path):
    """examples/c_caller.c: the drop-in surface from C (single call + batch), on a packed input written by the format oracle."""
    import subprocess

    from fhe_precompiles_b200 import pack

    a, b = encrypt_value(keys, "i64", 16, 1101), encrypt_value(keys, "i64", 4, 1102)
    packed = pack.pack_binary_operation(keys.pub_bytes, F.make_ciphertext("i64", a).to_bytes(), F.make_ciphertext("i64", b).to_bytes())
    (tmp_path / "in.bin").write_bytes(packed)
    exe = tmp_path / "c_caller"
    lib_dir = os.path.join(ROOT, "fhe_precompiles_b200")
    subprocess.run(["gcc", "-std=c11", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "c_caller.c"), "-L" + lib_dir,
                    "-lfhe_precompiles_b200", "-Wl,-rpath," + lib_dir, "-o", str(exe)], check=True)
    env = dict(os.environ, FHE_B200_ZSTD_WRITER="structured" if STRUCT() else "seal")
    r = subprocess.run([str(exe), str(tmp_path / "in.bin")], capture_output=True, text=True, timeout=300, env=env)
    want = len(F.make_ciphertext("i64", bfv.mul_relin(a, b, keys.rk)).to_bytes(structured=STRUCT()))
    assert r.returncode == 0, r.stdout + r.stderr
    assert f"result ciphertext: {want} bytes" in r.stdout and f"batch: 0 failed, outputs {want} and {want} bytes" in r.stdout, r.stdout


def test_uncompressed_operands_echo_their_compr_mode(keys):
    """SEAL blobs with compr_mode none are legal inputs (Serialization::Load reads any mode); the result echoes the mode of the
    ciphertext operand. Such calls bypass the device codec (single call and inside a tile) and go through the host pass."""
    from fhe_precompiles_b200 import FHE, pack

    a, b = encrypt_value(keys, "u64", 9, 1001), encrypt_value(keys, "u64", 5, 1002)
    raw_a = F.make_ciphertext("u64", a).to_bytes(compr=F.COMPR_NONE)
    raw_b = F.make_ciphertext("u64", b).to_bytes(compr=F.COMPR_NONE)
    z_b = F.make_ciphertext("u64", b).to_bytes()
    want_mul = F.make_ciphertext("u64", bfv.mul_relin(a, b, keys.rk))
    want_sub = F.make_ciphertext("u64", bfv.sub(a, b))
    p_raw = pack.pack_binary_operation(keys.pub_bytes, raw_a, raw_b)
    p_mixed = pack.pack_binary_operation(keys.pub_bytes, raw_a, z_b)  # the first operand's mode is echoed
    for packed in (p_raw, p_mixed):
        assert FHE.mul_cipheru64_cipheru64(packed) == want_mul.to_bytes(compr=F.COMPR_NONE)
        assert FHE.sub_cipheru64_cipheru64(packed) == want_sub.to_bytes(compr=F.COMPR_NONE)
    p_z = pack.pack_binary_operation(keys.pub_bytes, F.make_ciphertext("u64", a).to_bytes(), z_b)
    res = FHE.run_batch([("mul_cipheru64_cipheru64", p_raw), ("mul_cipheru64_cipheru64", p_z), ("sub_cipheru64_cipheru64", p_mixed),
                         ("mul_cipheru64_cipheru64", p_z)], host_threads=1)
    assert res == [(0, want_mul.to_bytes(compr=F.COMPR_NONE)), (0, want_mul.to_bytes(structured=STRUCT())),
                   (0, want_sub.to_bytes(compr=F.COMPR_NONE)), (0, want_mul.to_bytes(structured=STRUCT()))]
    assert decrypt_value(keys, "u64", F.Ciphertext.from_bytes(res[0][1]).polys()) == 45
    # zlib mode (compr_mode 1) is echoed too
    zl_a = F.make_ciphertext("u64", a).to_bytes(compr=F.COMPR_ZLIB)
    out = FHE.mul_cipheru64_cipheru64(pack.pack_binary_operation(keys.pub_bytes, zl_a, z_b))
    got = F.Ciphertext.from_bytes(out)
    assert np.array_equal(got.polys(), want_mul.polys()) and out == want_mul.to_bytes(compr=F.COMPR_ZLIB)


def test_batches_and_single_calls_concurrently(keys):
    """tiles (device codec, shared lanes, host pool) and single calls (fast path, CUDA-graph replay) from several threads at
    once; every result must equal the oracle's bytes."""
    import threading

    from fhe_precompiles_b200 import FHE, pack

    a, b = encrypt_value(keys, "i64", 11, 901), encrypt_value(keys, "i64", -4, 902)
    sa = F.make_ciphertext("i64", a).to_bytes()
    sb = F.make_ciphertext("i64", b).to_bytes(structured=True)
    pm = pack.pack_binary_operation(keys.pub_bytes, sa, sb)
    pn = pack.pack_binary_operation(keys.net_pub_bytes, sa, sb)
    ps = pack.pack_binary_operation(keys.pub_bytes, sa, pack.serialize_i64(3))
    want = {
        "mul": F.make_ciphertext("i64", bfv.mul_relin(a, b, keys.rk)).to_bytes(structured=STRUCT()),
        "mul_net": F.make_ciphertext("i64", bfv.mul_relin(a, b, keys.net_rk)).to_bytes(structured=STRUCT()),
        "add": F.make_ciphertext("i64", bfv.add(a, b)).to_bytes(structured=STRUCT()),
        "mulp": F.make_ciphertext("i64", bfv.multiply_plain(a, bfv.encode("i64", 3))).to_bytes(structured=STRUCT()),
    }
    batch = [("mul_cipheri64_cipheri64", pm), ("add_cipheri64_cipheri64", pm), ("mul_cipheri64_i64", ps),
             ("mul_cipheri64_cipheri64", pn), ("sub_cipheri64_cipheri64", b"\x00")] * 5
    batch_want = [want["mul"], want["add"], want["mulp"], want["mul_net"], None] * 5
    errors = []

    def batches(tid):
        try:
            for _ in range(4):
                res = FHE.run_batch(batch, host_threads=3)
                for (st, out), w in zip(res, batch_want):
                    if (w is None and st != 1) or (w is not None and (st != 0 or out != w)):
                        errors.append(("batch", tid, st))
        except Exception as e:  # noqa: BLE001
            errors.append(("batch", tid, repr(e)))

    def singles(tid):
        try:
            for it in range(24):
                which = ("mul", "add", "mulp", "mul_net")[(tid + it) % 4]
                if which == "mul":
                    out = FHE.mul_cipheri64_cipheri64(pm)
                elif which == "add":
                    out = FHE.add_cipheri64_cipheri64(pm)
                elif which == "mulp":
                    out = FHE.mul_cipheri64_i64(ps)
                else:
                    out = FHE.mul_cipheri64_cipheri64(pn)
                if out != want[which]:
                    errors.append(("single", tid, which))
        except Exception as e:  # noqa: BLE001
            errors.append(("single", tid, repr(e)))

    threads = [threading.Thread(target=batches, args=(i,)) for i in range(2)] + [threading.Thread(target=singles, args=(i,)) for i in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors[:5]


def test_second_device_and_cross_device_batch(dev, keys):
    """per-device contexts: the same kernels on cuda:1 (own twiddles / constants / key copies) and a byte-surface batch whose
    calls are spread over every GPU. Skipped on single-GPU boxes."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from fhe_precompiles_b200 import FHE, pack

    dev.init(1)
    a, b = edge_ct(3, 31), edge_ct(3, 32)[::-1].copy()
    want = np.stack([bfv.mul_relin(x, y, keys.rk) for x, y in zip(a, b)])
    t1 = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.int64)).to("cuda:1")
    with torch.cuda.device(1):
        got = dev.mul_relin(t1(a), t1(b), t1(keys.rk)).cpu().numpy().view(np.uint64)
        x = np.random.default_rng(1).integers(0, MODULI[4], size=(3, N), dtype=np.uint64)
        d = t1(x)
        dev.ntt_(d, [4])
        assert np.array_equal(d.cpu().numpy().view(np.uint64), bfv.ntt_fwd(x, 4))
    assert np.array_equal(got, want)
    ca, cb = encrypt_value(keys, "i64", 9, 1), encrypt_value(keys, "i64", -5, 2)
    sa, sb = (F.make_ciphertext("i64", c).to_bytes() for c in (ca, cb))
    packed = pack.pack_binary_operation(keys.pub_bytes, sa, sb)
    wm = F.make_ciphertext("i64", bfv.mul_relin(ca, cb, keys.rk)).to_bytes(structured=STRUCT())
    res = FHE.run_batch([("mul_cipheri64_cipheri64", packed)] * 24, host_threads=8)
    assert all(st == 0 and out == wm for st, out in res)


def test_mul_relin_frames_matches_oracle(dev, keys):
    """fhe_b200_mul_relin_frames: serialized operands (structured zstd frames) in, structured frames out, through the three-slot
    pipeline (more ops than one pipeline chunk).  Result frames are byte-identical to the format oracle's frames of the oracle's
    products; a frame that is not the structured layout and a residue >= q are flagged (status 1) without disturbing neighbours."""
    import torch

    n, bad_layout, bad_range = 300, 7, 123
    # one corrupted FIXED byte per frame (frame header, block headers, literal headers, sequence sections): what any zstd decoder
    # -- and so SEAL -- would reject or read differently must never come back with status 0
    bad_header = {20: 4, 21: 5, 22: 9, 23: 12, 24: 14 + 110 + 1, 25: 14 + 110 + 6, 26: 9 + 122, 27: 9 + 122 + 3, 28: 82054 - 7, 29: 82054 - 1}
    cts_a, cts_b = random_ct(np.random.default_rng(41), n), random_ct(np.random.default_rng(42), n)  # (constant polynomials are not
    # written as structured frames by any writer: they take the status-1 route like the libzstd frame below)
    fb_, fs = dev.frame_bytes(), dev.frame_stride()
    stride = fs + 32  # any stride >= the frame size works (e.g. whole packed ciphertexts)

    def frames_of(cts):
        buf = np.zeros((n, stride), dtype=np.uint8)
        for i in range(n):
            fr = F.zstd_structured_frame(F.fresh_data_ciphertext(cts[i]).payload())
            assert fr is not None and len(fr) == fb_
            buf[i, :fb_] = np.frombuffer(fr, dtype=np.uint8)
        return buf

    fa, fbuf = frames_of(cts_a), frames_of(cts_b)
    lib_frame = F.zstd().compress(F.fresh_data_ciphertext(cts_a[bad_layout]).payload())  # a libzstd frame: valid zstd, not structured
    fa[bad_layout, :] = 0
    fa[bad_layout, : min(len(lib_frame), stride)] = np.frombuffer(lib_frame[:stride], dtype=np.uint8)
    over = cts_b[bad_range].copy()
    over[0, 0, 5] = MODULI[0]  # residue == q0
    fbuf[bad_range, :fb_] = np.frombuffer(F.zstd_structured_frame(F.fresh_data_ciphertext(over).payload()), dtype=np.uint8)

    assert fb_ == 82054
    for i, off in bad_header.items():
        (fa if i & 1 else fbuf)[i, off] ^= 0x10

    ta, tb = torch.from_numpy(fa).pin_memory(), torch.from_numpy(fbuf).pin_memory()
    out = torch.zeros((n, fs), dtype=torch.uint8).pin_memory()
    status = torch.full((n,), -1, dtype=torch.int32).pin_memory()
    rk = torch.from_numpy(keys.rk.view(np.int64))
    dev.mul_relin_frames(ta, tb, rk, out, status)
    st = status.numpy()
    assert st[bad_layout] == 1 and st[bad_range] == 1
    assert all(st[i] == 1 for i in bad_header), [int(st[i]) for i in bad_header]
    ok = [i for i in range(n) if i not in (bad_layout, bad_range) and i not in bad_header]
    assert (st[ok] == 0).all()
    for i in ok[:6] + ok[250:262] + ok[-4:]:
        want = F.zstd_structured_frame(F.fresh_data_ciphertext(bfv.mul_relin(cts_a[i], cts_b[i], keys.rk)).payload())
        assert out[i, :fb_].numpy().tobytes() == want, f"result frame {i} differs from the oracle's"


# ---------------------------------------------------------------- round 2: encryptor parity, noise budget, exact types, configs 4 / 5
# the reference's private 512-bit constant mixed into the encrypt seed (fhe.rs:604-609)
SEED_CONSTANT = bytes([15, 17, 225, 5, 30, 1, 237, 218, 130, 19, 37, 95, 222, 218, 244, 172, 214, 175, 175, 110, 173, 103, 172, 60, 43,
                       76, 40, 150, 215, 96, 23, 78, 22, 39, 30, 177, 107, 130, 124, 109, 27, 96, 206, 125, 104, 241, 10, 40, 88, 238,
                       117, 118, 79, 113, 213, 110, 148, 179, 53, 19, 227, 154, 151, 122])


def seed_words(msg: bytes) -> np.ndarray:
    """u8_bits_to_u64_512_bits(SHA-512(msg)) (fhe.rs:47-54, 611)"""
    import hashlib

    return np.frombuffer(hashlib.sha512(msg).digest(), dtype="<u8").copy()


def test_device_encrypt_matches_oracle(dev, keys):
    """fhe_b200_encrypt against the oracle's restatement of sunscreen's encrypt_deterministic (Blake2xb PRNG, libstdc++
    ternary + clipped-normal samplers, data-level encryption; pinned by the reference's known answers): bit-exact, all kinds."""
    import torch

    rng = np.random.default_rng(91)
    vals = [("i64", -12345), ("i64", 2**62 + 17), ("u64", 2**64 - 1), ("u256", 2**255 + 9), ("frac64", -2.75), ("frac64", 1e9 + 0.5),
            ("i64", 0), ("u64", 0)]
    n = len(vals)
    seeds = rng.integers(0, 2**63, size=(n, 8), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    seeds[0] = 0  # the all-zero seed is a seed like any other
    plains = np.stack([plain_u16(k, v) for k, v in vals])
    for pk_np in (keys.net_pk, keys.pk):
        ct = to_np(dev.encrypt(to_dev(pk_np), torch.from_numpy(plains.view(np.int16)).cuda(), to_dev(seeds)))
        for i, (k, v) in enumerate(vals):
            assert np.array_equal(ct[i], bfv.encrypt_seeded(pk_np, bfv.encode(k, v), seeds[i])), f"op {i} ({k} {v})"
    # one flipped seed bit anywhere in the 512 changes the samples
    base = to_np(dev.encrypt(to_dev(keys.net_pk), torch.from_numpy(plains[:1].view(np.int16)).cuda(), to_dev(seeds[1:2])))
    for word in range(8):
        s2 = seeds[1:2].copy()
        s2[0, word] ^= np.uint64(1) << np.uint64(63 if word % 2 else 0)
        other = to_np(dev.encrypt(to_dev(keys.net_pk), torch.from_numpy(plains[:1].view(np.int16)).cuda(), to_dev(s2)))
        assert not np.array_equal(other[0, 1], base[0, 1]), f"seed word {word} is ignored"


@pytest.mark.parametrize("kind,value", [("i64", -7), ("u64", 2**64 - 1), ("u256", 2**200 + 5), ("frac64", -2.75)])
def test_encrypt_and_reencrypt_bytes_match_oracle(keys, kind, value):
    """c_fhe_encrypt_* / c_fhe_reencrypt_* through the byte surface: seed = SHA-512 exactly as fhe.rs:600-611 and
    fhe.rs:646-649, 676 build it, handed to the GPU restatement of SEAL's sampler stack; bytes == the oracle's."""
    from fhe_precompiles_b200 import FHE, pack

    ser = pack.SERIALIZE[kind](value)
    public = bytes([9, 8, 7])
    enc = getattr(FHE, f"encrypt_{kind}")(pack.pack_two_arguments(ser, public))
    want = bfv.encrypt_seeded(keys.net_pk, bfv.encode(kind, value), seed_words(public + SEED_CONSTANT + ser))
    assert enc == F.make_ciphertext(kind, want).to_bytes(structured=STRUCT())
    packed = pack.pack_binary_operation(keys.pub_bytes, enc, public)
    re = getattr(FHE, f"reencrypt_{kind}")(packed)
    want2 = bfv.encrypt_seeded(keys.pk, bfv.encode(kind, value), seed_words(public + packed + ser))
    assert re == F.make_ciphertext(kind, want2).to_bytes(structured=STRUCT())
    assert decrypt_value(keys, kind, F.Ciphertext.from_bytes(re).polys()) == value_of(kind, value)


def test_reference_known_answers_through_the_c_abi(keys, writer_mode):
    """THE byte-level pin of the product: the reference's three SHA-512 known answers (fhe.rs:2083-2121 fhe_encrypt_test,
    2143-2185 fhe_refresh_test, 2188-2246 fhe_reencrypt_test; Linux values) reproduced by c_fhe_encrypt_u256 /
    c_fhe_reencrypt_u256 with the default (SEAL-bytes) writer -- PRNG, samplers, NTTs, scaling, decryption, serialisation and
    compression all on the product side, nothing from the oracle but the digests."""
    import hashlib

    from fhe_precompiles_b200 import FHE, pack
    from test_oracle_kat import KAT

    if writer_mode != "seal":
        pytest.skip("the known answers hash SEAL's compressed bytes")
    value, public = pack.SERIALIZE["u256"](12), bytes([1, 2, 3])
    enc = FHE.encrypt_u256(pack.pack_two_arguments(value, public))
    assert hashlib.sha512(enc).digest() == bytes(KAT[("encrypt", "libstdc++")]), "fhe_encrypt_test"
    assert FHE.decrypt_u256(enc) == value
    # fhe_refresh_test: encrypt_deterministic(12, network key, seed = 0) re-encrypted under the network key
    ct0 = F.make_ciphertext("u256", bfv.encrypt_seeded(keys.net_pk, bfv.encode("u256", 12), bytes(64))).to_bytes()
    re0 = FHE.reencrypt_u256(pack.pack_binary_operation(keys.net_pub_bytes, ct0, public))
    assert hashlib.sha512(re0).digest() == bytes(KAT[("refresh", "libstdc++")]), "fhe_refresh_test"
    # fhe_reencrypt_test: the first result re-encrypted under tests/data/public_key.bin
    re1 = FHE.reencrypt_u256(pack.pack_binary_operation(keys.pub_bytes, enc, public))
    assert hashlib.sha512(re1).digest() == bytes(KAT[("reencrypt", "libstdc++")]), "fhe_reencrypt_test"
    assert decrypt_value(keys, "u256", F.Ciphertext.from_bytes(re1).polys()) == 12


def test_device_sampler_rare_paths(dev, keys):
    """the sampler's exact sequential paths: seeds whose stream has a zero draw inside u (Lemire redraw) cannot be found by
    search, but every seed exercises the compaction; a sweep of 64 seeds against the oracle covers attempts windows of
    different lengths, and the all-ones / all-zero seeds are seeds like any other."""
    import torch

    rng = np.random.default_rng(4242)
    n = 64
    seeds = rng.integers(0, 2**63, size=(n, 8), dtype=np.uint64)
    seeds[0] = 0
    seeds[1] = np.uint64(2**64 - 1)
    plains = np.zeros((n, N), dtype=np.uint16)
    plains[:, 0] = np.arange(n)
    ct = to_np(dev.encrypt(to_dev(keys.net_pk), torch.from_numpy(plains.view(np.int16)).cuda(), to_dev(seeds)))
    for i in range(n):
        assert np.array_equal(ct[i], bfv.encrypt_seeded(keys.net_pk, plains[i, :1].astype(np.uint64), seeds[i])), f"seed {i}"


def test_device_sampler_exact_paths_on_crafted_draws(dev):
    """k_seal_sample against the oracle's samplers on the SAME draws, including what no searchable seed reaches: a zero draw
    inside u (Lemire's redraw shifts every later draw by one), a clipped variate in e0 and in e1 (|3.2 z| > 19.2: it is
    dropped and everything behind it moves up), both together, a clipped variate as the very last sample, and draws that
    run out (failed = 1)."""
    import hashlib

    import torch

    ndraw = 28 * 1024
    base = [np.frombuffer(bfv.seal_prng(hashlib.sha512(b"crafted %d" % i).digest(), 4 * ndraw), dtype="<u4").copy() for i in range(8)]
    # an attempt whose first variate is clipped: x = 0 exactly (canonical = 1/2), y = 1e-4 -> r2 = 1e-8, sqrt(-2 ln r2) = 6.07
    y_hi = 0x80000000 + int(1e-4 * 2**31)
    clip = np.array([0, 0x80000000, 0, y_hi], dtype=np.uint32)
    cases = [base[0].copy()]
    z = base[1].copy(); z[100] = 0; z[4000] = 0; cases.append(z)                       # two redraws in u
    c = base[2].copy(); c[4096 + 4 * 50: 4096 + 4 * 50 + 4] = clip; cases.append(c)     # clipped variate early in e0
    c = base[3].copy(); c[4096 + 4 * 4000: 4096 + 4 * 4000 + 4] = clip; cases.append(c)  # ... in e1's range
    c = base[4].copy(); c[7] = 0; c[4097 + 4 * 10: 4097 + 4 * 10 + 4] = clip; cases.append(c)  # both (attempts start at 4097)
    c = base[5].copy(); c[4096: 4096 + 4000] = np.tile(clip, 1000); cases.append(c)    # e0's first 1,000 attempts all clip once
    c = base[6].copy(); c[4096:] = 0xFFFFFFFF; cases.append(c)                          # every attempt rejected: draws run out
    cases.append(base[7].copy())
    draws = torch.from_numpy(np.stack(cases).view(np.int32)).cuda()
    u, e0, e1, failed = (t.cpu().numpy() for t in dev.seal_sample(draws))
    for i, w in enumerate(cases):
        wu, we0, we1, drawn = bfv.seal_sample_stream(w)
        assert bool(failed[i]) == (drawn == 0), f"case {i}: failed flag"
        if drawn:
            assert np.array_equal(u[i], wu) and np.array_equal(e0[i], we0) and np.array_equal(e1[i], we1), f"case {i}"
    assert list(failed) == [0, 0, 0, 0, 0, 0, 1, 0]
    # the crafted cases really took the rare paths
    assert not np.array_equal(bfv.seal_sample_stream(base[1])[0], u[1]) and not np.array_equal(bfv.seal_sample_stream(base[2])[1], e0[2])
    assert (e0[5][:1000] == 0).all() and e0[5][1000:].any()  # only the second variate (x * mult = 0) of those attempts survives


def test_qlimb_recovery_equals_seals_form(dev, keys):
    """Both forms of multiply + relinearise -- chunks >= 96 ops (fused tails, key switch on the dual base) and smaller chunks
    (split tails, key switch on SEAL's key primes) -- through mul_relin and through multiply followed by relinearize: same
    bits on random and on extreme residues, equal to the oracle (which follows SEAL)."""
    import hashlib

    rng = np.random.default_rng(606)
    a, b = random_ct(rng, 128), random_ct(rng, 128)
    for l in range(2):
        a[20, :, l, :] = MODULI[l] - 1; b[20, :, l, :] = MODULI[l] - 1      # every coefficient q-1: the largest |t D|
        a[21, :, l, :] = MODULI[l] // 2; b[21, :, l, :] = MODULI[l] // 2 + 1
    a[22] = 0; b[23] = 0
    want = np.stack([bfv.mul_relin(a[i], b[i], keys.rk) for i in range(128)])
    sha = lambda x: hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()
    da, db, drk = to_dev(a), to_dev(b), to_dev(keys.rk)
    shas = {}
    prev = dev.set_chunk_ops(0)
    try:
        for chunk in (4096, 64):  # the default: one chunk of 128 ops; then two chunks of 64
            dev.set_chunk_ops(chunk)
            shas[chunk, "mul_relin"] = sha(to_np(dev.mul_relin(da, db, drk)))
            shas[chunk, "multiply + relinearize"] = sha(to_np(dev.relinearize(dev.multiply(da, db), drk)))
    finally:
        dev.set_chunk_ops(prev)
    assert shas == {k: sha(want) for k in shas}


def test_exhausted_noise_budget_is_failed_decryption(dev, keys):
    """sunscreen's Runtime::decrypt refuses a ciphertext whose invariant noise budget is 0 (-> FailedDecryption = 5,
    fhe.rs:640-643, 692-696).  Three multiplications deep there is none left at these parameters (53 -> 30 -> 7 -> 0 bits);
    the byte surface still multiplies such operands happily (as the reference does), but decrypt_* and reencrypt_* must return
    5, not a garbage scalar."""
    import torch

    from fhe_precompiles_b200 import FHE, FheError, pack

    cts = [encrypt_value(keys, "i64", v, 40 + i, network=True) for i, v in enumerate((3, 5, 7, 11))]
    p1 = bfv.mul_relin(cts[0], cts[1], keys.net_rk)
    p2 = bfv.mul_relin(cts[2], cts[3], keys.net_rk)
    p12 = bfv.mul_relin(p1, p2, keys.net_rk)   # 1155, 7 bits of budget left
    deep = bfv.mul_relin(p12, p1, keys.net_rk)  # exhausted
    budgets = [bfv.decrypt(c, keys.net_sk)[1] for c in (cts[0], p1, p12, deep)]
    assert budgets[0] > 40 and budgets[1] > 20 and 0 < budgets[2] < 12 and budgets[3] <= 0, budgets
    plain, flags = dev.decrypt_checked(to_dev(np.stack([cts[0], p1, deep, p12])), to_dev(keys.net_sk))
    assert flags.cpu().tolist() == [0, 0, 1, 0]
    assert bfv.decode("i64", plain[1].cpu().numpy().view(np.uint16).astype(np.uint64)) == 15
    assert bfv.decode("i64", plain[3].cpu().numpy().view(np.uint16).astype(np.uint64)) == 1155
    ser = lambda c: F.make_ciphertext("i64", c).to_bytes()
    assert pack.deserialize_scalar("i64", FHE.decrypt_i64(ser(p1))) == 15
    with pytest.raises(FheError) as e:
        FHE.decrypt_i64(ser(deep))
    assert e.value.code == 5
    with pytest.raises(FheError) as e:
        FHE.reencrypt_i64(pack.pack_binary_operation(keys.pub_bytes, ser(deep), b"\x01"))
    assert e.value.code == 5
    # the over-multiplied ciphertext is still a valid OPERAND (the reference's add/mul never look at the budget)
    out = FHE.add_cipheri64_cipheri64(pack.pack_binary_operation(keys.net_pub_bytes, ser(deep), ser(p1)))
    assert F.Ciphertext.from_bytes(out).polys().shape == (2, 2, N)


def test_argument_type_check_follows_sunscreens_type_names(keys):
    """sunscreen compares an argument's Type (name, version, is_encrypted) with the program's signature -> code 7 on a mismatch
    (fhe.rs:28).  `#[derive(TypeName)]` drops generic arguments, so Unsigned64 and Unsigned256 ciphertexts carry the SAME name
    (pinned by the reference's known answers, which hash it) and are interchangeable in the reference; a Signed ciphertext in an
    unsigned precompile, a foreign type, another crate version or is_encrypted = false are mismatches -- in single calls and
    inside batch tiles, for every operand position."""
    from fhe_precompiles_b200 import FHE, FheError, pack

    a64, b256 = encrypt_value(keys, "u64", 5, 1), encrypt_value(keys, "u256", 9, 2)
    c64 = F.make_ciphertext("u64", a64).to_bytes()
    c256 = F.make_ciphertext("u256", b256).to_bytes()
    ci64 = F.make_ciphertext("i64", encrypt_value(keys, "i64", 5, 3)).to_bytes()
    assert F.data_type_string("u64") == F.data_type_string("u256") == "sunscreen::types::bfv::unsigned::Unsigned,0.8.1,true"
    s64, s256 = pack.serialize_u64(3), pack.serialize_u256(3)

    def retag(blob, dt):
        c = F.Ciphertext.from_bytes(blob)
        c.data_type = dt
        return c.to_bytes()

    # interchangeable widths: the results are the plain ciphertext arithmetic
    out = FHE.add_cipheru256_cipheru256(pack.pack_binary_operation(keys.pub_bytes, c64, c256))
    assert out == F.make_ciphertext("u256", bfv.add(a64, b256)).to_bytes(structured=STRUCT())
    out = FHE.mul_cipheru64_cipheru64(pack.pack_binary_operation(keys.pub_bytes, c256, c64))
    assert out == F.make_ciphertext("u64", bfv.mul_relin(b256, a64, keys.rk)).to_bytes(structured=STRUCT())
    assert decrypt_value(keys, "u64", F.Ciphertext.from_bytes(out).polys()) == 45
    enc = FHE.encrypt_u64(pack.pack_two_arguments(s64, b"x"))
    assert FHE.decrypt_u256(enc) == s256
    bad = [
        ("add_cipheru64_cipheru64", (ci64, c64)), ("add_cipheru256_cipheru256", (c256, ci64)), ("add_cipheri64_cipheri64", (c64, c64)),
        ("mul_u64_cipheru64", (s64, ci64)), ("sub_cipheru256_u256", (ci64, s256)),
        ("add_cipheru64_cipheru64", (retag(c64, "sunscreen::types::bfv::rational::Rational,0.8.1,true"), c64)),
        ("add_cipheru64_cipheru64", (retag(c64, "sunscreen::types::bfv::unsigned::Unsigned,0.8.0,true"), c64)),
        ("add_cipheru64_cipheru64", (c64, retag(c64, "sunscreen::types::bfv::unsigned::Unsigned,0.8.1,false"))),
        ("add_cipheru64_cipheru64", (retag(c64, "sunscreen::types::bfv::unsigned::Unsigned<1>,0.8.1,true"), c64)),
        ("add_cipherfrac64_cipherfrac64", (c64, c64)),
    ]
    calls = []
    for name, (x, y) in bad:
        data = pack.pack_binary_operation(keys.pub_bytes, x, y)
        calls.append((name, data))
        with pytest.raises(FheError) as e:
            getattr(FHE, name)(data)
        assert e.value.code == 7, name
    good = ("add_cipheru64_cipheru64", pack.pack_binary_operation(keys.pub_bytes, c64, c256))
    res = FHE.run_batch(calls + [good] + calls, host_threads=2)
    assert [r[0] for r in res] == [7] * len(bad) + [0] + [7] * len(bad)
    # decrypt_* of another kind: FailedDecryption (fhe.rs:696)
    with pytest.raises(FheError) as e:
        FHE.decrypt_i64(enc)
    assert e.value.code == 5


SCALAR_EDGES = {
    "i64": [0, 1, -1, 2**63 - 1, -(2**63), -5, 12345],
    "u64": [0, 1, 2**64 - 1, 2**63],
    "u256": [0, 1, 2**256 - 1, 2**255, 2**128 + 3],
    "frac64": [0.0, 1.0, -1.0, 0.5, -0.375, 2.0**40 + 0.25, 1.0 / 3.0, -123456.789],
}


@pytest.mark.parametrize("kind", KINDS)
def test_scalar_edge_cases_through_the_c_abi(keys, kind):
    """ct o pt and pt o ct with edge scalars (0 -> transparent product accepted, negative, extreme, fractions): result
    bytes == oracle, and the decrypted value equals the plain arithmetic in the type's own wrap-around."""
    from fhe_precompiles_b200 import FHE, pack

    base = {"i64": -3, "u64": 7, "u256": 2**130 + 1, "frac64": 1.5}[kind]
    ct = encrypt_value(keys, kind, base, 77)
    ser_ct = F.make_ciphertext(kind, ct).to_bytes()
    calls, wants = [], []
    for v in SCALAR_EDGES[kind]:
        for op in ("add", "sub", "mul"):
            for shape in ("ctpt", "ptct"):
                sc = pack.SERIALIZE[kind](v)
                args, oargs = ((ser_ct, sc), (ct, v)) if shape == "ctpt" else ((sc, ser_ct), (v, ct))
                calls.append((precompile_name(op, shape, kind), pack.pack_binary_operation(keys.pub_bytes, *args)))
                wants.append(oracle_binary(op, shape, kind, *oargs, keys.rk))
    res = FHE.run_batch(calls)
    for (name, data), (st, out), want in zip(calls, res, wants):
        assert st == 0, name
        assert out == F.make_ciphertext(kind, want).to_bytes(structured=STRUCT()), name  # (constant results fall back to libzstd in both)
    # single calls give the same bytes (spot check incl. the transparent case, fhe.rs:2124-2140)
    for i in (0, 1, 4, len(calls) - 1):
        assert getattr(FHE, calls[i][0])(calls[i][1]) == res[i][1]
    # decrypted values: the mul-by-0 result is all-zero (transparent) and decrypts to 0
    k0 = [i for i, (name, _) in enumerate(calls) if name.startswith("mul")][0]
    assert not F.Ciphertext.from_bytes(res[k0][1]).polys().any()
    wrap = {"i64": lambda x: (x + 2**63) % 2**64 - 2**63, "u64": lambda x: x % 2**64, "u256": lambda x: x % 2**256, "frac64": float}[kind]
    j = 0
    for v in SCALAR_EDGES[kind]:
        for op in ("add", "sub", "mul"):
            for shape in ("ctpt", "ptct"):
                x, y = (base, v) if shape == "ctpt" else (v, base)
                exact = {"add": x + y, "sub": x - y, "mul": x * y}[op]
                got = decrypt_value(keys, kind, F.Ciphertext.from_bytes(res[j][1]).polys())
                if kind == "frac64":
                    assert abs(got - exact) <= 1e-9 * max(1.0, abs(exact)), (calls[j][0], v)  # f64 rounding of the encoder only
                else:
                    assert got == wrap(exact), (calls[j][0], v)
                j += 1


def test_large_batch_device_decoder_equals_small_batches(keys):
    """fhe_b200_batch on a batch large enough for the default big tiles + device zstd decoder (>= 2,048 calls: operand frames
    inflated by k_zd2_parse / k_zd3_seq / k_zd3_exec) against the same calls in 16-call batches (operands inflated by libzstd
    on the host): 2,304 ct.ct calls over 96 distinct uniformly random ciphertexts (libzstd level-3 frames), some corrupted;
    every status and every output byte equal."""
    import ctypes

    from fhe_precompiles_b200 import FHE, _lib, pack

    L = _lib.lib()
    rng = np.random.default_rng(77)
    dt = b"sunscreen::types::bfv::signed::Signed,0.8.1,true"

    def blob() -> bytes:
        w = np.stack([rng.integers(0, MODULI[l], N, dtype=np.uint64) for _ in range(2) for l in range(2)]).reshape(-1)
        out, ln = ctypes.c_void_p(), ctypes.c_int64()
        assert L.fhe_b200_write_ciphertext(w.ctypes.data, dt, ctypes.byref(out), ctypes.byref(ln)) == 0
        b = ctypes.string_at(out.value, ln.value)
        L.fhe_free(out)
        return b

    prev = L.fhe_b200_set_zstd_writer(0)  # operands as SEAL writes them
    try:
        cts = [blob() for _ in range(96)]
    finally:
        L.fhe_b200_set_zstd_writer(prev)
    calls = []
    for i in range(2304):
        a, b = cts[int(rng.integers(96))], cts[int(rng.integers(96))]
        if i % 97 == 13:  # a flipped bit somewhere in the first operand's frame: the device decoder or the range check hands it back
            bad = bytearray(a)
            bad[-int(rng.integers(1, 80000))] ^= 1 << int(rng.integers(8))
            a = bytes(bad)
        op = ("mul", "add", "sub")[i % 3]
        calls.append((f"{op}_cipheri64_cipheri64", pack.pack_binary_operation(keys.pub_bytes, a, b)))
    big = FHE.run_batch(calls)
    small = []
    for k in range(0, len(calls), 16):
        small += FHE.run_batch(calls[k : k + 16], host_threads=2)
    assert [g[0] for g in big] == [w[0] for w in small]
    assert sum(1 for st, _ in big if st == 0) >= 2200
    assert all(g[1] == w[1] for g, w in zip(big, small))


def test_config4_mixed_batch_matches_oracle(keys):
    """BASELINE config 4 at one GPU's share: 4,608 calls drawn (seed 3) uniformly from {add, sub, mul} x {ct.ct, ct.pt, pt.ct}
    x {u64, i64, u256, frac64} -- every one of the 36 precompiles many times -- through fhe_b200_batch in tiles; EVERY result
    byte-compared with the oracle's.  Operands come from a pool of 24 ciphertexts per kind (half libzstd level-3 frames as
    SEAL writes them, half structured frames) so that the expected values stay a few thousand oracle calls."""
    from fhe_precompiles_b200 import FHE, pack

    rng = np.random.default_rng(3)
    pool_n, n_calls = 24, 4608
    vals = {"u64": lambda i: 3 + 5 * i, "i64": lambda i: (-1) ** i * (7 + i), "u256": lambda i: 2**100 + i, "frac64": lambda i: 0.5 * i - 3.25}
    pool = {k: [encrypt_value(keys, k, value_of(k, vals[k](i)), 2000 + 100 * ki + i) for i in range(pool_n)] for ki, k in enumerate(KINDS)}
    ser = {k: [F.make_ciphertext(k, c).to_bytes(structured=bool(i & 1)) for i, c in enumerate(pool[k])] for k in KINDS}
    scal = {k: [value_of(k, vals[k](i + 1)) for i in range(6)] for k in KINDS}
    calls, keys_of = [], []
    cache = {}
    for _ in range(n_calls):
        op = ("add", "sub", "mul")[rng.integers(3)]
        shape = SHAPES[rng.integers(3)]
        kind = KINDS[rng.integers(4)]
        i, j = int(rng.integers(pool_n)), int(rng.integers(pool_n if shape == "ctct" else 6))
        if shape == "ctct":
            args, oargs = (ser[kind][i], ser[kind][j]), (pool[kind][i], pool[kind][j])
        elif shape == "ctpt":
            args, oargs = (ser[kind][i], pack.SERIALIZE[kind](scal[kind][j])), (pool[kind][i], scal[kind][j])
        else:
            args, oargs = (pack.SERIALIZE[kind](scal[kind][j]), ser[kind][i]), (scal[kind][j], pool[kind][i])
        key = (op, shape, kind, i, j)
        if key not in cache:
            cache[key] = (pack.pack_binary_operation(keys.pub_bytes, *args), oargs)
        calls.append((precompile_name(op, shape, kind), cache[key][0]))
        keys_of.append(key)
    assert len({c[0] for c in calls}) == 36
    res = FHE.run_batch(calls)
    assert all(st == 0 for st, _ in res)
    want_bytes = {}
    for key, (st, out) in zip(keys_of, res):
        if key not in want_bytes:
            op, shape, kind = key[:3]
            w = oracle_binary(op, shape, kind, *cache[key][1], keys.rk)
            want_bytes[key] = F.make_ciphertext(kind, w).to_bytes(structured=STRUCT())
        assert out == want_bytes[key], key


def test_config5_encrypt_decrypt_roundtrip(dev, keys):
    """BASELINE config 5 at one GPU's share of 16,384: pk-encrypt 2,048 random i64 under network.pub on the GPU, decrypt with
    network.pri, all equal, no ciphertext flagged as exhausted; 32 ciphertexts bit-compared with the oracle's encryptor."""
    import torch

    n = 2048
    rng = np.random.default_rng(5)
    vals = rng.integers(-(2**62), 2**62, size=n)
    mag = np.abs(vals).astype(np.uint64)
    bits = ((mag[:, None] >> np.arange(64, dtype=np.uint64)[None, :]) & 1).astype(np.int64)
    plains = np.zeros((n, N), dtype=np.uint16)
    plains[:, :64] = np.where(vals[:, None] < 0, bits * 4095, bits).astype(np.uint16)
    seeds = rng.integers(0, 2**63, size=(n, 8), dtype=np.uint64)
    ct = dev.encrypt(to_dev(keys.net_pk), torch.from_numpy(plains.view(np.int16)).cuda(), to_dev(seeds))
    plain, flags = dev.decrypt_checked(ct, to_dev(keys.net_sk))
    assert not flags.any()
    assert np.array_equal(plain.cpu().numpy().view(np.uint16), plains)
    cts = to_np(ct)
    for i in range(0, n, 64):
        assert np.array_equal(cts[i], bfv.encrypt_seeded(keys.net_pk, plains[i, :64].astype(np.uint64), seeds[i])), f"op {i}"


def test_upload_chain_download_frames(dev, keys):
    """Serialized ciphertexts -> device-resident limb arrays -> a chain of device-resident ops -> serialized result: PCIe is crossed
    once at each end.  300 ciphertexts (two transfer chunks); result frames byte-identical to the format oracle's frames of the
    oracle's (a * b + a) - b; a frame with a corrupted fixed byte, a residue >= q and a non-structured frame are rejected
    (status 1); a transparent result has no structured frame (status 2)."""
    import torch

    n = 300
    rng = np.random.default_rng(61)
    a, b = random_ct(rng, n), random_ct(rng, n)
    fb_, fs = dev.frame_bytes(), dev.frame_stride()
    stride = fs + 8

    def frames_of(cts):
        buf = np.zeros((len(cts), stride), dtype=np.uint8)
        for i, c in enumerate(cts):
            buf[i, :fb_] = np.frombuffer(F.zstd_structured_frame(F.fresh_data_ciphertext(c).payload()), dtype=np.uint8)
        return buf

    fa, fbuf = frames_of(a), frames_of(b)
    bad = {5: "fixed byte", 17: "range", 200: "libzstd frame"}
    fa[5, 10] ^= 0x40
    over = a[17].copy()
    over[1, 1, 4095] = MODULI[1]
    fa[17, :fb_] = np.frombuffer(F.zstd_structured_frame(F.fresh_data_ciphertext(over).payload()), dtype=np.uint8)
    lib_frame = F.zstd().compress(F.fresh_data_ciphertext(a[200]).payload())
    fa[200, :] = 0
    fa[200, :] = np.frombuffer(lib_frame[:stride], dtype=np.uint8)
    da, sa = dev.upload_frames(torch.from_numpy(fa).pin_memory())
    db, sb = dev.upload_frames(torch.from_numpy(fbuf))  # pageable memory works too
    assert sb.tolist() == [0] * n
    assert [i for i in range(n) if sa[i] != 0] == sorted(bad) and all(sa[i] == 1 for i in bad)
    ok = [i for i in range(n) if i not in bad]
    assert np.array_equal(to_np(da)[ok], a[ok]) and np.array_equal(to_np(db), b)
    rk = to_dev(keys.rk)
    res = dev.sub(dev.add(dev.mul_relin(da, db, rk), da), db)
    out, st = dev.download_frames(res)
    assert st.tolist() == [0] * n
    for i in ok[:4] + [255, 256, 257, n - 1]:
        want = bfv.sub(bfv.add(bfv.mul_relin(a[i], b[i], keys.rk), a[i]), b[i])
        assert out[i, :fb_].numpy().tobytes() == F.zstd_structured_frame(F.fresh_data_ciphertext(want).payload()), f"ciphertext {i}"
    # round trip of the frames themselves, and a transparent ciphertext
    back, st2 = dev.download_frames(db)
    assert st2.tolist() == [0] * n and np.array_equal(back[:, :fb_].numpy(), fbuf[:, :fb_])
    _, st3 = dev.download_frames(dev.sub(db[:3], db[:3]))
    assert st3.tolist() == [2, 2, 2]
