"""Threshold precompiles (encrypt_*, reencrypt_*, decrypt_*) through fhe_b200_batch, and the per-row-key device encryption
their tiles use: every status and every output byte equals the single c_fhe_* call's, and the rows equal the oracle's."""
import ctypes
import hashlib

import numpy as np
import pytest

from helpers import KINDS, MODULI, N, decrypt_value, encrypt_value, value_of
from oracle import bfv
from oracle import formats as F
from test_oracle_kat import SEED_CONSTANT

pytestmark = pytest.mark.gpu

VALUES = {"u256": 2**200 + 5, "u64": 2**64 - 1, "i64": -7, "frac64": -2.75}


@pytest.fixture(params=["seal", "structured"])
def writer(request):
    """the result writer: "seal" (libzstd level 3, SEAL's bytes, the default) or "structured" (frames written on the GPU)"""
    from fhe_precompiles_b200 import _lib

    L = _lib.lib()
    prev = L.fhe_b200_set_zstd_writer(1 if request.param == "structured" else 0)
    yield request.param
    L.fhe_b200_set_zstd_writer(prev)


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


def seed_words(msg: bytes) -> np.ndarray:
    return np.frombuffer(hashlib.sha512(msg).digest(), dtype="<u8").copy()


def single(name: str, data: bytes):
    from fhe_precompiles_b200 import FHE, FheError

    try:
        return (0, getattr(FHE, name)(data))
    except FheError as e:
        return (e.code, b"")


def run_indexed(calls, host_threads: int = 0):
    """fhe_b200_batch on (op index, bytes) pairs, so that an index outside the op table can be passed too"""
    from fhe_precompiles_b200 import _lib

    L = _lib.lib()
    arr = (_lib.BatchCall * len(calls))()
    keep = []
    for i, (idx, data) in enumerate(calls):
        buf = (ctypes.c_char * max(len(data), 1)).from_buffer_copy(data or b"\0")
        keep.append(buf)
        arr[i].op, arr[i].bytes, arr[i].bytes_length = idx, ctypes.cast(buf, ctypes.c_void_p), len(data)
    L.fhe_b200_batch(arr, len(calls), host_threads)
    res = []
    for c in arr:
        res.append((c.status, ctypes.string_at(c.output, c.output_length) if c.status == 0 else b""))
        if c.status == 0:
            L.fhe_free(c.output)
    return res


# ---------------------------------------------------------------- 1. device encryption with a key per row
def test_encrypt_keyed_row_for_row(dev):
    """fhe_b200_encrypt_keyed: row i equals fhe_b200_encrypt under pks[key_index[i]] for every index pattern (all 0, round
    robin, random, one row per key), equals the oracle on every 64th row, and is the same when the rows span several chunks."""
    import torch

    rng = np.random.default_rng(314)
    n, k = 2048, 5
    pks = np.empty((k, 2, 3, N), dtype=np.uint64)
    for l in range(3):
        pks[:, :, l, :] = rng.integers(0, MODULI[l], size=(k, 2, N), dtype=np.uint64)
    plains = rng.integers(0, 4096, size=(n, N), dtype=np.uint16)
    seeds = rng.integers(0, 2**63, size=(n, 8), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    d_pks, d_plain, d_seeds = to_dev(pks), torch.from_numpy(plains.view(np.int16)).cuda(), to_dev(seeds)
    per_key = [to_np(dev.encrypt(d_pks[j].contiguous(), d_plain, d_seeds)) for j in range(k)]
    patterns = {
        "zeros": np.zeros(n, dtype=np.int32),
        "round robin": (np.arange(n) % k).astype(np.int32),
        "random": rng.integers(0, k, size=n).astype(np.int32),
    }
    for name, idx in patterns.items():
        got = to_np(dev.encrypt_keyed(d_pks, torch.from_numpy(idx).cuda(), d_plain, d_seeds))
        want = np.stack([per_key[idx[i]][i] for i in range(n)])
        assert np.array_equal(got, want), name
    idx = patterns["random"]
    for i in range(0, n, 64):
        assert np.array_equal(got[i], bfv.encrypt_seeded(pks[idx[i]], plains[i].astype(np.uint64), seeds[i])), f"row {i}"
    # one row per key, in an order that is not the keys'
    one = np.array([3, 0, 4, 1, 2], dtype=np.int32)
    got = to_np(dev.encrypt_keyed(d_pks, torch.from_numpy(one).cuda(), d_plain[:k].contiguous(), d_seeds[:k].contiguous()))
    assert all(np.array_equal(got[i], per_key[one[i]][i]) for i in range(k))
    # more rows than a chunk: the same bits
    prev = dev.set_chunk_ops(0)
    try:
        dev.set_chunk_ops(768)
        got = to_np(dev.encrypt_keyed(d_pks, torch.from_numpy(idx).cuda(), d_plain, d_seeds))
    finally:
        dev.set_chunk_ops(prev)
    assert np.array_equal(got, np.stack([per_key[idx[i]][i] for i in range(n)]))
    # no rows: nothing to do
    assert dev.encrypt_keyed(d_pks, torch.zeros(0, dtype=torch.int32).cuda(), d_plain[:0], d_seeds[:0]).shape == (0, 2, 2, N)


# ---------------------------------------------------------------- 2. batch == single calls, faults included
def threshold_calls(keys):
    """(name, bytes) of ~60 threshold calls over the four kinds and the three operations, operands as SEAL libzstd frames,
    structured frames and uncompressed blobs, with a fault at every stage"""
    from fhe_precompiles_b200 import pack

    calls = []
    public = bytes([4, 5, 6])
    for j, kind in enumerate(KINDS):
        v = VALUES[kind]
        ser = pack.SERIALIZE[kind](v)
        calls.append((f"encrypt_{kind}", pack.pack_two_arguments(ser, public)))
        calls.append((f"encrypt_{kind}", pack.pack_two_arguments(pack.SERIALIZE[kind](value_of(kind, 3 + j)), bytes([j]))))
        ct = F.make_ciphertext(kind, encrypt_value(keys, kind, v, 50 + j, network=True))
        for blob in (ct.to_bytes(), ct.to_bytes(structured=True), ct.to_bytes(compr=F.COMPR_NONE)):
            calls.append((f"decrypt_{kind}", pack.pack_one_argument(blob)))
            calls.append((f"reencrypt_{kind}", pack.pack_binary_operation(keys.pub_bytes, blob, public)))
        calls.append((f"reencrypt_{kind}", pack.pack_binary_operation(keys.net_pub_bytes, ct.to_bytes(), bytes([j, j]))))
    # faults: truncated framing (1), a key that does not parse (3), a ciphertext of another kind (5), a corrupt frame
    u256 = F.make_ciphertext("u256", encrypt_value(keys, "u256", 12, 60, network=True)).to_bytes()
    i64 = F.make_ciphertext("i64", encrypt_value(keys, "i64", -3, 61, network=True)).to_bytes()
    good = pack.pack_binary_operation(keys.pub_bytes, i64, public)
    calls.append(("encrypt_i64", b"\x00\x00"))
    calls.append(("reencrypt_i64", good[:11]))
    calls.append(("reencrypt_i64", good[:8] + b"junk" + good[12:]))
    calls.append(("decrypt_i64", u256))
    calls.append(("reencrypt_i64", pack.pack_binary_operation(keys.pub_bytes, u256, public)))
    bad = bytearray(i64)
    bad[-300] ^= 0x10
    calls.append(("decrypt_i64", bytes(bad)))
    calls.append(("reencrypt_i64", pack.pack_binary_operation(keys.pub_bytes, bytes(bad), public)))
    calls.append(("decrypt_i64", i64[:-9]))
    # an exhausted noise budget (5): three multiplications deep
    cts = [encrypt_value(keys, "i64", v, 40 + i, network=True) for i, v in enumerate((3, 5, 7, 11))]
    p1 = bfv.mul_relin(cts[0], cts[1], keys.net_rk)
    deep = bfv.mul_relin(bfv.mul_relin(p1, bfv.mul_relin(cts[2], cts[3], keys.net_rk), keys.net_rk), p1, keys.net_rk)
    deep_b = F.make_ciphertext("i64", deep).to_bytes()
    calls.append(("decrypt_i64", deep_b))
    calls.append(("reencrypt_i64", pack.pack_binary_operation(keys.pub_bytes, deep_b, public)))
    # a frac64 value that fails to encode (6), and a scalar of the wrong length (3)
    calls.append(("encrypt_frac64", pack.pack_two_arguments(pack.serialize_frac64(float("nan")), public)))
    calls.append(("encrypt_u64", pack.pack_two_arguments(b"\x01" * 5, public)))
    return calls


def test_batch_equals_single_calls(keys, writer):
    """~60 threshold calls mixed with binary calls, public_key_bytes and an op index outside the table: each status and output
    equals the single symbol's under either writer, for 1, 2 and 16 host threads and for a permutation of the calls."""
    from fhe_precompiles_b200 import _lib, pack

    L = _lib.lib()
    calls = threshold_calls(keys)
    a = F.make_ciphertext("i64", encrypt_value(keys, "i64", 6, 70)).to_bytes()
    b = F.make_ciphertext("i64", encrypt_value(keys, "i64", 7, 71)).to_bytes(structured=True)
    binary = pack.pack_binary_operation(keys.pub_bytes, a, b)
    calls += [("mul_cipheri64_cipheri64", binary), ("add_cipheri64_cipheri64", binary), ("public_key_bytes", b"")]
    want = [single(name, data) for name, data in calls] + [(7, b"")]
    codes = {st for st, _ in want}
    assert {0, 1, 3, 5, 6, 7} <= codes, codes
    indexed = [(L.fhe_b200_op_index(name.encode()), data) for name, data in calls] + [(99, b"")]
    for threads in (1, 2, 16):
        got = run_indexed(indexed, threads)
        wrong = [i for i in range(len(want)) if got[i] != want[i]]
        assert not wrong, (threads, [(calls[i][0] if i < len(calls) else "op 99", got[i][0], want[i][0]) for i in wrong[:8]])
    perm = np.random.default_rng(5).permutation(len(indexed))
    got = run_indexed([indexed[i] for i in perm], 0)
    assert all(got[k] == want[perm[k]] for k in range(len(perm)))


def test_ordinary_calls_take_the_tile(keys, writer):
    """20 threshold calls whose operands are libzstd or structured frames of their kind: in 16-call tiles they launch a
    third of the kernels the same calls launch one by one (one decryption and one encryption per tile, not per call)."""
    from fhe_precompiles_b200 import _lib, pack

    L = _lib.lib()
    calls = []
    for j, kind in enumerate(KINDS):
        v = value_of(kind, 20 + j)
        ct = F.make_ciphertext(kind, encrypt_value(keys, kind, v, 80 + j, network=True))
        calls.append((f"encrypt_{kind}", pack.pack_two_arguments(pack.SERIALIZE[kind](v), bytes([j]))))
        for blob in (ct.to_bytes(), ct.to_bytes(structured=True)):
            calls.append((f"decrypt_{kind}", blob))
            calls.append((f"reencrypt_{kind}", pack.pack_binary_operation(keys.pub_bytes, blob, bytes([j]))))
    before = L.fhe_b200_launch_count()
    want = [single(name, data) for name, data in calls]
    single_launches = L.fhe_b200_launch_count() - before
    assert all(st == 0 for st, _ in want)
    before = L.fhe_b200_launch_count()
    got = run_indexed([(L.fhe_b200_op_index(name.encode()), data) for name, data in calls], 1)
    tile_launches = L.fhe_b200_launch_count() - before
    assert got == want
    assert 3 * tile_launches < single_launches, (tile_launches, single_launches)


ODD_LANES = r"""
import sys
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
from helpers import KeySet, encrypt_value, value_of
from oracle import formats as F
from fhe_precompiles_b200 import FHE, FheError, _lib, pack

def single(name, data):
    try:
        return (0, getattr(FHE, name)(data))
    except FheError as e:
        return (e.code, b"")

keys = KeySet.load()
ct = F.make_ciphertext("i64", encrypt_value(keys, "i64", -5, 7, network=True)).to_bytes()
a = F.make_ciphertext("i64", encrypt_value(keys, "i64", 6, 8)).to_bytes()
three = [("encrypt_i64", pack.pack_two_arguments(pack.serialize_i64(41), b"x")), ("decrypt_i64", ct),
         ("reencrypt_i64", pack.pack_binary_operation(keys.pub_bytes, ct, b"y"))]
binary = [(n, pack.pack_binary_operation(keys.pub_bytes, a, a)) for n in ("add_cipheri64_cipheri64", "sub_cipheri64_cipheri64",
                                                                          "mul_cipheri64_cipheri64")] * 3
threshold = [("encrypt_u64", pack.pack_two_arguments(pack.serialize_u64(i), bytes([i]))) for i in range(3)] + three[1:] * 2
mixed = [c for pair in zip(binary, threshold) for c in pair] + binary[len(threshold):]
L = _lib.lib()
for mode in (0, 1):
    L.fhe_b200_set_zstd_writer(mode)
    for batch in (three, mixed):  # lane 0 serves a 3-call tile, then a 9-call binary tile and a 7-call threshold tile
        got = FHE.run_batch(batch, host_threads=1)
        want = [single(n, d) for n, d in batch]
        assert got == want, (mode, len(batch), [g[0] for g in got], [w[0] for w in want])
        assert all(st == 0 for st, _ in got)
print("odd lanes ok")
"""


def test_threshold_tiles_on_lanes_of_odd_capacity():
    """Lanes grow to exactly the size of the largest tile they serve, so odd capacities are ordinary: in a fresh process lane 0
    serves a 3-call threshold tile, then a 16-call tile of 9 binary and 7 threshold calls, under either writer.  Every result
    equals the single call's (the per-lane key buffer of the encryption rows stays aligned whatever the capacity)."""
    import subprocess
    import sys

    from helpers import ROOT

    r = subprocess.run([sys.executable, "-c", ODD_LANES, ROOT], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "odd lanes ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ---------------------------------------------------------------- 3. big tiles
def test_big_tiles_equal_small_batches(dev, keys, writer):
    """2,112 threshold calls -- reencrypts of libzstd-written operands to four distinct target keys (the two real ones and two
    crafted: the same keys without their relinearisation keys) and decrypts -- run as big tiles whose operand frames the device
    decoder inflates.  Results equal the same calls in 16-call batches and, on sampled rows, the oracle's encryption under the
    row's own key; the launch counter shows batched launches."""
    from fhe_precompiles_b200 import FHE, pack

    bare = lambda pub: F.PublicKey(F.PublicKey.from_bytes(pub).public_key, None, None).to_bytes()
    targets = [(keys.pub_bytes, keys.pk), (keys.net_pub_bytes, keys.net_pk), (bare(keys.pub_bytes), keys.pk),
               (bare(keys.net_pub_bytes), keys.net_pk)]
    base, meta = [], []
    for i in range(24):
        kind = KINDS[i % 4]
        v = value_of(kind, 100 + i)
        ct = F.make_ciphertext(kind, encrypt_value(keys, kind, v, 900 + i, network=True)).to_bytes()
        pub, pk = targets[i % 4]
        packed = pack.pack_binary_operation(pub, ct, bytes([i]))
        base.append((f"reencrypt_{kind}", packed))
        meta.append((kind, v, pk, packed, bytes([i])))
        if i % 3 == 0:
            base.append((f"decrypt_{kind}", ct))
            meta.append(None)
    n = 2112
    batch = [base[i % len(base)] for i in range(n)]
    want = []
    for lo in range(0, len(base), 16):
        want += FHE.run_batch(base[lo: lo + 16])
    assert all(st == 0 for st, _ in want)
    before = dev.launch_count()
    got = FHE.run_batch(batch)
    launches = dev.launch_count() - before
    wrong = [i for i in range(n) if got[i] != want[i % len(base)]]
    assert not wrong, [(i, got[i][0]) for i in wrong[:8]]
    assert launches < n / 8, launches  # a single call launches at least five kernels
    structured = writer == "structured"
    for j in range(0, len(base), 5):
        if meta[j] is None:
            continue
        kind, v, pk, packed, public = meta[j]
        ser = pack.SERIALIZE[kind](v)
        row = bfv.encrypt_seeded(pk, bfv.encode(kind, v), seed_words(public + packed + ser))
        assert want[j][1] == F.make_ciphertext(kind, row).to_bytes(structured=structured), j


# ---------------------------------------------------------------- 4. the reference's known answers through the batch
def test_reference_known_answers_through_the_batch(keys):
    """fhe_encrypt_test, fhe_refresh_test and fhe_reencrypt_test (fhe.rs:2083-2246) with the default writer, as three calls of
    a 64-call batch whose tiles run them with other threshold calls."""
    from fhe_precompiles_b200 import FHE, _lib, pack
    from test_oracle_kat import KAT

    L = _lib.lib()
    prev = L.fhe_b200_set_zstd_writer(0)
    try:
        value, public = pack.SERIALIZE["u256"](12), bytes([1, 2, 3])
        enc_in = pack.pack_two_arguments(value, public)
        enc = F.make_ciphertext("u256", bfv.encrypt_seeded(keys.net_pk, bfv.encode("u256", 12),
                                                           seed_words(public + SEED_CONSTANT + value))).to_bytes()
        ct0 = F.make_ciphertext("u256", bfv.encrypt_seeded(keys.net_pk, bfv.encode("u256", 12), bytes(64))).to_bytes()
        kat = [("encrypt_u256", enc_in), ("reencrypt_u256", pack.pack_binary_operation(keys.net_pub_bytes, ct0, public)),
               ("reencrypt_u256", pack.pack_binary_operation(keys.pub_bytes, enc, public))]
        filler = [(f"encrypt_{k}", pack.pack_two_arguments(pack.SERIALIZE[k](value_of(k, i)), bytes([i]))) for i in range(61)
                  for k in (KINDS[i % 4],)]
        batch = filler[:5] + kat[:1] + filler[5:9] + kat[1:2] + filler[9:12] + kat[2:] + filler[12:]
        res = FHE.run_batch(batch, host_threads=1)
        pos = [batch.index(c) for c in kat]
        assert all(res[p][0] == 0 for p in pos)
        assert res[pos[0]][1] == enc
        assert hashlib.sha512(res[pos[0]][1]).digest() == bytes(KAT[("encrypt", "libstdc++")]), "fhe_encrypt_test"
        assert hashlib.sha512(res[pos[1]][1]).digest() == bytes(KAT[("refresh", "libstdc++")]), "fhe_refresh_test"
        assert hashlib.sha512(res[pos[2]][1]).digest() == bytes(KAT[("reencrypt", "libstdc++")]), "fhe_reencrypt_test"
        assert all(r == single(name, data) for r, (name, data) in zip(res, batch))
    finally:
        L.fhe_b200_set_zstd_writer(prev)


# ---------------------------------------------------------------- 5. round trips
def test_round_trips_through_the_batch(keys, writer):
    """encrypt -> reencrypt to tests/data/public_key.bin -> decrypt with private_key.bin (oracle) gives the value back for every
    kind; encrypt -> decrypt_* in the batch too."""
    from fhe_precompiles_b200 import FHE, pack

    vals = [(k, v) for k in KINDS for v in (VALUES[k], value_of(k, 12), value_of(k, 0))]
    enc = FHE.run_batch([(f"encrypt_{k}", pack.pack_two_arguments(pack.SERIALIZE[k](v), bytes([7]))) for k, v in vals])
    assert all(st == 0 for st, _ in enc)
    calls = [(f"reencrypt_{k}", pack.pack_binary_operation(keys.pub_bytes, ct, b"rt")) for (k, _), (_, ct) in zip(vals, enc)]
    calls += [(f"decrypt_{k}", ct) for (k, _), (_, ct) in zip(vals, enc)]
    res = FHE.run_batch(calls)
    m = len(vals)
    for j, (k, v) in enumerate(vals):
        assert res[j][0] == 0 and decrypt_value(keys, k, F.Ciphertext.from_bytes(res[j][1]).polys()) == value_of(k, v), (k, v)
        assert res[m + j][0] == 0 and pack.deserialize_scalar(k, res[m + j][1]) == value_of(k, v), (k, v)
