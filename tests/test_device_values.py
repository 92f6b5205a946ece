"""Device-resident typed values: fhe_b200_encode_values / fhe_b200_decode_values and device.encode / decode / encrypt_values /
decrypt_values, bit-compared with the oracle's encoders and with the byte surface (c_fhe_*) on the same values.
Bar: bit-exact, frac64 included (compared as the 8 bytes of the double).  Run on the B200 box: pytest -m gpu."""
import ctypes
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

from helpers import KINDS, N, ROOT, encrypt_value, plain_u16, random_ct
from oracle import bfv
from oracle import formats as F
from test_oracle_kat import SEED_CONSTANT

pytestmark = pytest.mark.gpu

M64 = 2**64 - 1
I64_MIN, I64_MAX = -(2**63), 2**63 - 1
EDGES = {
    "i64": [0, 1, -1, I64_MIN, I64_MAX, -7, 12],
    "u64": [0, 1, M64, 12, 2**63],
    "u256": [0, 1, 2**255, 2**256 - 1, 2**200 + 5, 12],
    "frac64": [0.0, -0.0, 5e-324, 2.2250738585072014e-308, 1e-300, -2.75, 1e9 + 0.5, 2.0**63, float(np.nextafter(2.0**64, 0.0)),
               -float(np.nextafter(2.0**64, 0.0)), 12.0, -1e-310],
}
OUT_OF_RANGE = [2.0**64, -(2.0**64), float("inf"), float("-inf"), float("nan"), 1e300]


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


def random_values(kind: str, rng: np.random.Generator, n: int) -> list:
    if kind == "frac64":
        mant = rng.standard_normal(n)
        return [float(m * 10.0 ** int(e)) for m, e in zip(mant, rng.integers(-320, 19, n))]
    bits = {"u64": 64, "i64": 64, "u256": 256}[kind]
    vals = [int.from_bytes(rng.bytes(bits // 8), "little") for _ in range(n)]
    return [v - 2**63 if kind == "i64" else v for v in vals]


def values_tensor(kind: str, vals):
    import torch

    if kind == "frac64":
        return torch.tensor(np.array(vals, dtype=np.float64)).cuda()
    if kind == "u256":
        w = np.array([[(int(v) >> (64 * k)) & M64 for k in range(4)] for v in vals], dtype=np.uint64).reshape(len(vals), 4)
        return torch.from_numpy(w.view(np.int64)).cuda()
    a = np.array([int(v) & M64 for v in vals], dtype=np.uint64) if kind == "u64" else np.array(vals, dtype=np.int64)
    return torch.from_numpy(a.view(np.int64)).cuda()


def comparable(kind: str, v):
    """a value in a form that compares bit for bit: ints, and the 8 bytes of a double"""
    return struct.pack("<d", float(v)) if kind == "frac64" else int(v)


def device_values(kind: str, t) -> list:
    a = t.cpu().numpy()
    if kind == "frac64":
        return [comparable(kind, x) for x in a]
    if kind == "u256":
        w = a.view(np.uint64)
        return [sum(int(w[i, k]) << (64 * k) for k in range(4)) for i in range(w.shape[0])]
    return [int(x) for x in (a.view(np.uint64) if kind == "u64" else a)]


def oracle_decode(kind: str, row: np.ndarray):
    return comparable(kind, bfv.decode(kind, row.astype(np.uint64)))


def assert_decodes_like_oracle(dev, kind, plains: np.ndarray, what: str):
    import torch

    got = device_values(kind, dev.decode(kind, torch.from_numpy(plains.astype(np.uint16).view(np.int16)).cuda()))
    for i, row in enumerate(plains):
        assert got[i] == oracle_decode(kind, row), f"{kind} {what} row {i}"


# ---------------------------------------------------------------- encode
@pytest.mark.parametrize("kind", KINDS)
def test_encode_matches_oracle(dev, kind):
    rng = np.random.default_rng(31 + KINDS.index(kind))
    vals = EDGES[kind] + random_values(kind, rng, 200)
    plain, status = dev.encode(kind, values_tensor(kind, vals))
    got = plain.cpu().numpy().view(np.uint16)
    assert not status.cpu().numpy().any()
    for i, v in enumerate(vals):
        assert np.array_equal(got[i], plain_u16(kind, v)), f"{kind} {v!r}"


def test_encode_frac64_out_of_range_is_status_7(dev):
    vals = [1.5] + OUT_OF_RANGE + [-2.75]
    plain, status = dev.encode("frac64", values_tensor("frac64", vals))
    got = plain.cpu().numpy().view(np.uint16)
    assert status.cpu().tolist() == [0] + [7] * len(OUT_OF_RANGE) + [0]
    for i in range(1, 1 + len(OUT_OF_RANGE)):
        assert not got[i].any(), vals[i]
        with pytest.raises(ValueError):
            bfv.encode("frac64", vals[i])  # the oracle refuses the same values
    assert np.array_equal(got[0], plain_u16("frac64", 1.5)) and np.array_equal(got[-1], plain_u16("frac64", -2.75))


def test_encode_status_may_be_null(dev):
    import torch

    from fhe_precompiles_b200 import _lib

    vals = values_tensor("i64", [-5, 9])
    plain = torch.empty((2, N), dtype=torch.int16, device="cuda")
    assert _lib.lib().fhe_b200_encode_values(0, 2, vals.data_ptr(), plain.data_ptr(), None, 2, None) == 0
    torch.cuda.synchronize()
    assert np.array_equal(plain.cpu().numpy().view(np.uint16), np.stack([plain_u16("i64", -5), plain_u16("i64", 9)]))


# ---------------------------------------------------------------- decode
@pytest.mark.parametrize("kind", KINDS)
def test_decode_matches_oracle(dev, kind):
    rng = np.random.default_rng(41 + KINDS.index(kind))
    encoded = np.stack([plain_u16(kind, v) for v in EDGES[kind] + random_values(kind, rng, 40)])
    full = rng.integers(0, 2**16, size=(48, N), dtype=np.uint64)
    below_t = rng.integers(0, 4096, size=(48, N), dtype=np.uint64)
    edge = np.zeros((6, N), dtype=np.uint64)
    edge[1], edge[2], edge[3], edge[4] = 4095, 2048, 2047, 65535
    edge[5, ::7] = 4096  # c == t: the magnitude t - c is 0
    # frac64's subnormal / underflow bands: sparse rows around indices 2990..3140
    bands = np.zeros((48, N), dtype=np.uint64)
    for r in range(48):
        idx = rng.integers(2980, 3150, size=24)
        bands[r, idx] = rng.integers(0, 2**16 if r % 2 else 4096, size=24)
        bands[r, rng.integers(0, 64, size=3)] = rng.integers(0, 4096, size=3)
    for what, plains in (("encoding", encoded), ("full-range", full), ("< t", below_t), ("edge", edge), ("band", bands)):
        assert_decodes_like_oracle(dev, kind, plains, what)


@pytest.mark.parametrize("kind", KINDS)
def test_decode_of_decrypted_products(dev, keys, kind):
    """the plaintexts a real chain ends in: decryptions of mul_relin products of real encryptions (dense low coefficients)"""
    rng = np.random.default_rng(51 + KINDS.index(kind))
    if kind == "frac64":
        va = [float(x) for x in rng.uniform(-1e6, 1e6, 8)]
        vb = [float(x) for x in rng.uniform(-1e3, 1e3, 8)]
    else:
        va = [int(x) for x in rng.integers(0 if kind != "i64" else -(2**30), 2**30, 8)]
        vb = [int(x) for x in rng.integers(1, 2**30, 8)]
    a = np.stack([encrypt_value(keys, kind, v, 7000 + i) for i, v in enumerate(va)])
    b = np.stack([encrypt_value(keys, kind, v, 7100 + i) for i, v in enumerate(vb)])
    prod = dev.mul_relin(to_dev(a), to_dev(b), to_dev(keys.rk))
    plains = dev.decrypt(prod, to_dev(keys.sk)).cpu().numpy().view(np.uint16)
    assert_decodes_like_oracle(dev, kind, plains, "product")
    values, exhausted = dev.decrypt_values(prod, to_dev(keys.sk), kind)
    assert not exhausted.cpu().numpy().any()
    assert device_values(kind, values) == [oracle_decode(kind, p) for p in plains]
    if kind != "frac64":
        want = [(x * y) % 2**64 if kind != "u256" else x * y for x, y in zip(va, vb)]
        got = device_values(kind, values)
        assert [g % 2**64 for g in got] == [w % 2**64 for w in want]


# ---------------------------------------------------------------- byte-surface parity
def seed_words(msg: bytes) -> np.ndarray:
    import hashlib

    return np.frombuffer(hashlib.sha512(msg).digest(), dtype="<u8").copy()


def write_ciphertext(words: np.ndarray, kind: str) -> bytes:
    from fhe_precompiles_b200 import _lib

    L = _lib.lib()
    w = np.ascontiguousarray(words, dtype=np.uint64)
    out, n = ctypes.c_void_p(), ctypes.c_int64()
    assert L.fhe_b200_write_ciphertext(w.ctypes.data, F.data_type_string(kind).encode(), ctypes.byref(out), ctypes.byref(n)) == 0
    try:
        return ctypes.string_at(out.value, n.value)
    finally:
        L.fhe_free(out)


@pytest.mark.parametrize("kind", KINDS)
def test_encrypt_and_decrypt_values_match_the_byte_surface(dev, keys, kind):
    """encrypt_values with the byte surface's seed (SHA-512(public | constant | serialized value)) writes the bytes of
    c_fhe_encrypt_<kind>; decrypt_values of those ciphertexts and of c_fhe_* results gives c_fhe_decrypt_<kind>'s values."""
    import torch

    from fhe_precompiles_b200 import FHE, pack

    vals = EDGES[kind]
    public = bytes([9, 8, 7])
    sers = [pack.SERIALIZE[kind](v) for v in vals]
    seeds = np.stack([seed_words(public + SEED_CONSTANT + s) for s in sers])
    ct, status = dev.encrypt_values(to_dev(keys.net_pk), kind, values_tensor(kind, vals), to_dev(seeds))
    assert not status.cpu().numpy().any()
    words = to_np(ct)
    encs = [getattr(FHE, f"encrypt_{kind}")(pack.pack_two_arguments(s, public)) for s in sers]
    for i, v in enumerate(vals):
        assert write_ciphertext(words[i], kind) == encs[i], f"{kind} {v!r}"
    # results of the byte surface's own arithmetic on those ciphertexts (under the network key, so c_fhe_decrypt reads them)
    three = pack.SERIALIZE[kind](3.0 if kind == "frac64" else 3)
    results = list(encs)
    for i in range(1, len(encs)):
        results.append(getattr(FHE, f"add_cipher{kind}_cipher{kind}")(pack.pack_binary_operation(keys.net_pub_bytes, encs[i - 1], encs[i])))
        results.append(getattr(FHE, f"mul_cipher{kind}_{kind}")(pack.pack_binary_operation(keys.net_pub_bytes, encs[i], three)))
    cts = torch.from_numpy(np.stack([F.Ciphertext.from_bytes(r).polys() for r in results]).astype(np.uint64).view(np.int64)).cuda()
    got, exhausted = dev.decrypt_values(cts, to_dev(keys.net_sk), kind)
    assert not exhausted.cpu().numpy().any()
    want = [comparable(kind, pack.deserialize_scalar(kind, getattr(FHE, f"decrypt_{kind}")(pack.pack_one_argument(r)))) for r in results]
    assert device_values(kind, got) == want


SCALAR_EDGES = {"u256": [2**255, 2**256 - 1], "u64": [M64, 1], "i64": [I64_MIN, -1], "frac64": [-2.75, 1e9 + 0.5, 1e-300]}
MODES = {("add", "ctpt"): 0, ("add", "ptct"): 0, ("sub", "ctpt"): 1, ("sub", "ptct"): 3}


@pytest.mark.parametrize("kind", KINDS)
def test_encode_then_plain_ops_match_all_scalar_precompiles(dev, keys, kind):
    """encode + plain_addsub (mode 0 add, 1 ct - pt, 3 pt - ct) / multiply_plain on a parsed ciphertext equals the words of
    c_fhe_{add,sub,mul}_{cipherT_T, T_cipherT}: the six scalar precompiles of each kind, on edge scalars."""
    import torch

    from fhe_precompiles_b200 import FHE, pack

    ct_bytes = F.make_ciphertext(kind, encrypt_value(keys, kind, 3 if kind != "frac64" else 3.5, 8100 + KINDS.index(kind))).to_bytes()
    ct_words = F.Ciphertext.from_bytes(ct_bytes).polys().astype(np.uint64)
    scalars = SCALAR_EDGES[kind]
    plain, status = dev.encode(kind, values_tensor(kind, scalars))
    assert not status.cpu().numpy().any()
    n = len(scalars)
    dct = to_dev(np.stack([ct_words] * n))
    for op in ("add", "sub", "mul"):
        for shape in ("ctpt", "ptct"):
            got = to_np(dev.multiply_plain(dct, plain) if op == "mul" else dev.plain_addsub(dct, plain, MODES[(op, shape)]))
            name = f"{op}_cipher{kind}_{kind}" if shape == "ctpt" else f"{op}_{kind}_cipher{kind}"
            for i, s in enumerate(scalars):
                ser = pack.SERIALIZE[kind](s)
                args = (ct_bytes, ser) if shape == "ctpt" else (ser, ct_bytes)
                out = getattr(FHE, name)(pack.pack_binary_operation(keys.pub_bytes, *args))
                assert np.array_equal(got[i], F.Ciphertext.from_bytes(out).polys().astype(np.uint64)), f"{name} {s!r}"


# ---------------------------------------------------------------- exhausted ciphertexts, batches, errors
def test_decrypt_values_flags_what_decrypt_checked_flags(dev, keys):
    rng = np.random.default_rng(61)
    real = np.stack([encrypt_value(keys, "i64", int(v), 9000 + i) for i, v in enumerate(rng.integers(-1000, 1000, 6))])
    cts = to_dev(np.concatenate([random_ct(rng, 10), real]))
    plain, flags = dev.decrypt_checked(cts, to_dev(keys.sk))
    flags = flags.cpu().numpy()
    assert flags[:10].all() and not flags[10:].any()  # uniform residues have no budget; fresh encryptions do
    for kind in KINDS:
        values, exhausted = dev.decrypt_values(cts, to_dev(keys.sk), kind)
        assert np.array_equal(exhausted.cpu().numpy(), flags), kind
        assert device_values(kind, values) == device_values(kind, dev.decode(kind, plain)), kind


def test_large_batch(dev):
    """100,000 rows in one launch (more than a grid dimension of 65,535 could index), checked on a sample including the last"""
    import torch

    n = 100_000
    g = torch.Generator(device="cuda").manual_seed(71)
    plain = torch.randint(-(2**15), 2**15, (n, N), dtype=torch.int16, device="cuda", generator=g)
    rows = sorted(set(np.random.default_rng(72).integers(0, n, 40).tolist()) | {0, 65_535, 65_536, n - 1})
    sample = plain[rows].cpu().numpy().view(np.uint16)
    for kind in KINDS:
        got = device_values(kind, dev.decode(kind, plain)[rows])
        assert got == [oracle_decode(kind, r) for r in sample], kind
    vals = random_values("i64", np.random.default_rng(73), n)
    enc, status = dev.encode("i64", values_tensor("i64", vals))
    assert not status.any().item()
    enc = enc[rows].cpu().numpy().view(np.uint16)
    for j, r in enumerate(rows):
        assert np.array_equal(enc[j], plain_u16("i64", vals[r])), r


def test_empty_batches_and_unknown_kinds(dev):
    import torch

    from fhe_precompiles_b200 import _lib

    L = _lib.lib()
    for kind in KINDS:
        plain, status = dev.encode(kind, values_tensor(kind, []))
        assert plain.shape == (0, N) and status.shape == (0,)
        assert dev.decode(kind, torch.empty((0, N), dtype=torch.int16, device="cuda")).shape[0] == 0
    launches = dev.launch_count()
    assert L.fhe_b200_encode_values(0, 1, None, None, None, 0, None) == 0
    assert L.fhe_b200_decode_values(0, 3, None, None, 0, None) == 0
    assert dev.launch_count() == launches  # n == 0 launches nothing
    for k in (-1, 4, 99):
        assert L.fhe_b200_encode_values(0, k, None, None, None, 1, None) == -1
        assert f"fhe_b200_encode_values: unknown kind {k}" in _lib.last_error()
        assert L.fhe_b200_decode_values(0, k, None, None, 1, None) == -1
        assert f"fhe_b200_decode_values: unknown kind {k}" in _lib.last_error()
    with pytest.raises(ValueError, match="unknown value kind"):
        dev.encode("u128", values_tensor("u64", [1]))
    with pytest.raises(ValueError, match="unknown value kind"):
        dev.decode("f32", torch.zeros((1, N), dtype=torch.int16, device="cuda"))


NO_DEVICE = r"""
import sys
sys.path.insert(0, sys.argv[1])
import torch
assert not torch.cuda.is_available()
from fhe_precompiles_b200 import _lib
L = _lib.lib()
assert L.fhe_b200_encode_values(0, 1, None, None, None, 1, None) == -1
assert L.fhe_b200_decode_values(0, 3, None, None, 1, None) == -1
assert "no CPU fallback" in _lib.last_error()
print("ok")
"""


def test_no_device_fails():
    r = subprocess.run([sys.executable, "-c", NO_DEVICE, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr
