"""Multiply + relinearise with a relinearisation key per row: the keyed device ops (fhe_b200_mul_relin_keyed,
fhe_b200_relinearize_keyed) row for row, and fhe_b200_batch tiles whose ct-ct multiplies belong to many users -- every status
and output byte equals the single c_fhe_* call's, and the tile launches one multiply sequence whatever the number of keys."""
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import KINDS, N, ROOT, decrypt_value, encrypt_value, precompile_name, random_ct, value_of
from oracle import bfv
from oracle import formats as F
from user_keys import KEY_MODULI, user_keys

pytestmark = pytest.mark.gpu

# kernels of one multiply + relinearise sequence (kernels.cu): ext_conv, ext_ntt, tensor_intt, floor_sk, digit_ntt, ks_intt,
# relin_finish below 96 ops; ext_conv, ext_ntt, tensor_floor, rk_intt_ksd, rk_lift_ksd, rk_ntt_ksd, digit_ntt_ksd, ks_tail_ksd
# from 96 on, the middle three being one group of prepared keys (7, 8 and 3 today).  sequence_launches() counts them on the
# device API, so that the tile launch test follows the sequence when it changes.
FUSED_TAIL_MIN_OPS = 96  # engine.cpp kFusedTailMinOps


@pytest.fixture(params=["seal", "structured"])
def writer(request):
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


@pytest.fixture(scope="module")
def users():
    return user_keys(64)


def to_dev(a: np.ndarray):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()


def to_np(t) -> np.ndarray:
    return t.cpu().numpy().view(np.uint64)


def random_keys(rng, k: int) -> np.ndarray:
    rks = np.empty((k, 2, 2, 3, N), dtype=np.uint64)
    for l, q in enumerate(KEY_MODULI):
        rks[:, :, :, l, :] = rng.integers(0, q, size=(k, 2, 2, N), dtype=np.uint64)
    return rks


def single(name: str, data: bytes):
    from fhe_precompiles_b200 import FHE, FheError

    try:
        return (0, getattr(FHE, name)(data))
    except FheError as e:
        return (e.code, b"")


# ---------------------------------------------------------------- 1. keyed device ops row for row
def per_key_rows(dev, fn, idx, d_rks, *ops):
    """row i of fn(*ops) under d_rks[idx[i]], one call per key over that key's rows"""
    import torch

    n = len(idx)
    out = np.empty((n, 2, 2, N), dtype=np.uint64)
    for j in np.unique(idx):
        rows = np.nonzero(idx == j)[0]
        sel = torch.from_numpy(rows).cuda()
        out[rows] = to_np(fn(*[o.index_select(0, sel).contiguous() for o in ops], d_rks[int(j)].contiguous()))
    return out


@pytest.mark.parametrize("n", [1, 95, 96, 97, 700])
def test_keyed_ops_row_for_row(dev, n):
    """mul_relin_keyed / relinearize_keyed: row i equals mul_relin / relinearize of that row under rks[key_index[i]] for all-zero,
    round-robin, random and one-key-per-row indices, at both tail forms and across their boundary; the oracle agrees on every
    64th row and on every row at n <= 97"""
    import torch

    rng = np.random.default_rng(700 + n)
    a, b = random_ct(rng, n), random_ct(rng, n)
    da, db = to_dev(a), to_dev(b)
    k = 5
    patterns = {
        "zeros": (np.zeros(n, dtype=np.int32), k),
        "round robin": ((np.arange(n) % k).astype(np.int32), k),
        "random": (rng.integers(0, k, size=n).astype(np.int32), k),
        "one key per row": (rng.permutation(n).astype(np.int32), n),
    }
    c3 = dev.multiply(da, db)
    for name, (idx, nk) in patterns.items():
        rks = random_keys(rng, nk)
        d_rks, d_idx = to_dev(rks), torch.from_numpy(idx).cuda()
        got = to_np(dev.mul_relin_keyed(da, db, d_rks, d_idx))
        assert np.array_equal(got, per_key_rows(dev, dev.mul_relin, idx, d_rks, da, db)), name
        got_r = to_np(dev.relinearize_keyed(c3, d_rks, d_idx))
        assert np.array_equal(got_r, got), name  # relinearize(multiply) is mul_relin, bit for bit
        rows = range(n) if n <= 97 else range(0, n, 64)
        for i in rows:
            assert np.array_equal(got[i], bfv.mul_relin(a[i], b[i], rks[idx[i]])), (name, i)


def test_keyed_ops_across_chunks(dev):
    """more keys than a chunk has ops, rows spread over several chunks (fused full chunks and a split last one, or split only):
    the same bits as one call per key"""
    import torch

    rng = np.random.default_rng(9)
    n, k = 700, 300
    a, b = random_ct(rng, n), random_ct(rng, n)
    da, db = to_dev(a), to_dev(b)
    rks = random_keys(rng, k)
    d_rks = to_dev(rks)
    idx = rng.integers(0, k, size=n).astype(np.int32)
    d_idx = torch.from_numpy(idx).cuda()
    want = per_key_rows(dev, dev.mul_relin, idx, d_rks, da, db)
    c3 = dev.multiply(da, db)
    prev = dev.set_chunk_ops(0)
    try:
        for chunk in (128, 64):
            dev.set_chunk_ops(chunk)
            assert np.array_equal(to_np(dev.mul_relin_keyed(da, db, d_rks, d_idx)), want), chunk
            assert np.array_equal(to_np(dev.relinearize_keyed(c3, d_rks, d_idx)), want), chunk
    finally:
        dev.set_chunk_ops(prev)
    for i in range(0, n, 64):
        assert np.array_equal(want[i], bfv.mul_relin(a[i], b[i], rks[idx[i]])), i


def test_keyed_ops_arguments(dev):
    """n == 0 launches nothing; wrong shapes or dtypes raise before anything reaches the device"""
    import torch

    rng = np.random.default_rng(3)
    rks = to_dev(random_keys(rng, 2))
    a = to_dev(random_ct(rng, 4))
    idx = torch.zeros(4, dtype=torch.int32).cuda()
    before = dev.launch_count()
    assert dev.mul_relin_keyed(a[:0], a[:0], rks, idx[:0]).shape == (0, 2, 2, N)
    assert dev.relinearize_keyed(torch.zeros((0, 3, 2, N), dtype=torch.int64).cuda(), rks, idx[:0]).shape == (0, 2, 2, N)
    assert dev.launch_count() == before
    bad = [
        (a, a, rks, idx.long()),  # int64 indices
        (a, a, rks[0], idx),  # one key without its key axis
        (a, a, rks, idx[:3]),  # an index short
        (a, a[:3], rks, idx),  # operands of different lengths
        (a.int(), a, rks, idx),  # int32 operands
    ]
    for args in bad:
        with pytest.raises((AssertionError, ValueError)):
            dev.mul_relin_keyed(*args)
    with pytest.raises((AssertionError, ValueError)):
        dev.relinearize_keyed(a, rks, idx)  # a size-2 ciphertext


# ---------------------------------------------------------------- 2. tiles equal single calls, many users
def user_calls(keys, users, n_users: int):
    """(name, bytes) of the 36 binary precompiles spread over n_users keys, operands as libzstd and structured frames, with
    faults: a truncated operand, a bit-flipped operand, an unparsable key, a key without relinearisation keys on a ct-ct multiply"""
    from fhe_precompiles_b200 import pack

    calls, meta = [], []
    u = 0
    # ct-ct multiplies, the calls whose key matters: user (7 i) mod n_users, spread over every tile of the batch
    muls, mul_meta = [], []
    for i in range(48):
        kind = KINDS[i % 4]
        pub, rk = users[(7 * i) % n_users]
        ca, cb = encrypt_value(keys, kind, value_of(kind, i), 1300 + i), encrypt_value(keys, kind, value_of(kind, 2), 1400 + i)
        sa = F.make_ciphertext(kind, ca).to_bytes(structured=i % 3 == 1)
        sb = F.make_ciphertext(kind, cb).to_bytes(structured=i % 3 == 2)
        muls.append((precompile_name("mul", "ctct", kind), pack.pack_binary_operation(pub, sa, sb)))
        mul_meta.append(("mul", "ctct", kind, ca, cb, rk))
    for op in ("mul", "add", "sub"):
        for shape in ("ctct", "ctpt", "ptct"):
            for j, kind in enumerate(KINDS):
                for structured in (False, True):
                    pub, rk = users[u % n_users]
                    u += 1
                    x, y = value_of(kind, 5 + j), value_of(kind, 3)
                    ca = encrypt_value(keys, kind, x, 300 + u)
                    cb = encrypt_value(keys, kind, y, 600 + u)
                    sa = F.make_ciphertext(kind, ca).to_bytes(structured=structured)
                    sb = F.make_ciphertext(kind, cb).to_bytes(structured=not structured)
                    left = sa if shape != "ptct" else pack.SERIALIZE[kind](x)
                    right = sb if shape == "ctct" else (pack.SERIALIZE[kind](y) if shape == "ctpt" else sa)
                    calls.append((precompile_name(op, shape, kind), pack.pack_binary_operation(pub, left, right)))
                    meta.append((op, shape, kind, ca, cb, rk) if shape == "ctct" and op == "mul" else None)
    # two multiplies after every three other calls
    mixed, mixed_meta = [], []
    for k in range(len(calls)):
        mixed.append(calls[k])
        mixed_meta.append(meta[k])
        if k % 3 == 2 and muls:
            mixed += muls[:2]
            mixed_meta += mul_meta[:2]
            del muls[:2], mul_meta[:2]
    calls, meta = mixed + muls, mixed_meta + mul_meta
    # faults
    pub, _ = users[1 % n_users]
    ca = F.make_ciphertext("i64", encrypt_value(keys, "i64", 9, 901)).to_bytes()
    cb = F.make_ciphertext("i64", encrypt_value(keys, "i64", 2, 902)).to_bytes()
    flipped = bytearray(cb)
    flipped[-300] ^= 0x10
    bare = F.PublicKey(F.PublicKey.from_bytes(pub).public_key, None, None).to_bytes()
    name = "mul_cipheri64_cipheri64"
    calls += [
        (name, pack.pack_binary_operation(pub, ca, cb[:-9])),
        (name, pack.pack_binary_operation(pub, ca, bytes(flipped))),
        (name, pack.pack_binary_operation(pub[:1000] + b"\xff" * 8 + pub[1008:], ca, cb)),
        (name, pack.pack_binary_operation(bare, ca, cb)),
        (name, pack.pack_binary_operation(bare, ca, cb[:-9])),
    ]
    meta += [None] * 5
    return calls, meta


@pytest.mark.parametrize("n_users", [16, 64])
def test_tiles_equal_single_calls(keys, users, writer, n_users):
    from fhe_precompiles_b200 import FHE

    calls, meta = user_calls(keys, users, n_users)
    want = [single(name, data) for name, data in calls]
    codes = {st for st, _ in want}
    assert 0 in codes and len(codes) >= 3, codes
    got = FHE.run_batch(calls, host_threads=4)  # 16-call tiles on four lanes
    wrong = [i for i in range(len(calls)) if got[i] != want[i]]
    assert not wrong, [(calls[i][0], got[i][0], want[i][0]) for i in wrong[:8]]
    perm = np.random.default_rng(n_users).permutation(len(calls))
    got = FHE.run_batch([calls[i] for i in perm], host_threads=1)
    assert all(got[k] == want[perm[k]] for k in range(len(perm)))
    structured = writer == "structured"
    for i in range(0, len(calls), 2):
        if meta[i] is None:
            continue
        _, _, kind, ca, cb, rk = meta[i]
        assert want[i][1] == F.make_ciphertext(kind, bfv.mul_relin(ca, cb, rk)).to_bytes(structured=structured), i


# ---------------------------------------------------------------- 3. big tiles
def big_batch(keys, users):
    from fhe_precompiles_b200 import pack

    kinds = ("i64", "u64")
    base, meta = [], []
    for u, (pub, rk) in enumerate(users):
        kind = kinds[u % 2]
        ca, cb = encrypt_value(keys, kind, value_of(kind, u), 2000 + u), encrypt_value(keys, kind, value_of(kind, 7), 3000 + u)
        packed = pack.pack_binary_operation(pub, F.make_ciphertext(kind, ca).to_bytes(), F.make_ciphertext(kind, cb).to_bytes())
        base.append((f"mul_cipher{kind}_cipher{kind}", packed))
        meta.append((kind, ca, cb, rk))
        if u % 8 == 0:
            base.append((f"add_cipher{kind}_cipher{kind}", packed))
            meta.append(None)
    return base, meta


BIG_BATCH = 2112

# the big batch in a fresh process whose key cache holds 4 keys: every tile misses, pins its keys past the capacity and evicts
# between tiles.  The batch runs, then 64 calls under 64 other users churn the cache, then the batch runs again.
SMALL_CACHE = r"""
import hashlib, json, sys
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
from helpers import KeySet, encrypt_value
from oracle import formats as F
from user_keys import user_key, user_keys
from test_multikey_batch import BIG_BATCH, big_batch
from fhe_precompiles_b200 import FHE, pack

keys = KeySet.load()
base, _ = big_batch(keys, user_keys(256))
batch = [base[i % len(base)] for i in range(BIG_BATCH)]
digest = lambda res: [[st, hashlib.sha256(out).hexdigest()] for st, out in res]
first = digest(FHE.run_batch(batch))
a = F.make_ciphertext("i64", encrypt_value(keys, "i64", 6, 8)).to_bytes()
churn = FHE.run_batch([("mul_cipheri64_cipheri64", pack.pack_binary_operation(user_key(1000 + j)[0], a, a)) for j in range(64)])
assert all(st == 0 for st, _ in churn)
second = digest(FHE.run_batch(batch))
json.dump({"first": first, "second": second}, open(sys.argv[2], "w"))
"""


def test_big_tiles_under_256_keys(dev, keys, writer):
    """2,112 calls, ct-ct multiplies under 256 user keys, run as big tiles whose operand frames the device decoder inflates:
    equal to the same calls in 16-call batches; sampled rows equal the oracle"""
    from fhe_precompiles_b200 import FHE

    users = user_keys(256)
    base, meta = big_batch(keys, users)
    want = []
    for lo in range(0, len(base), 16):
        want += FHE.run_batch(base[lo: lo + 16])
    assert all(st == 0 for st, _ in want)
    batch = [base[i % len(base)] for i in range(BIG_BATCH)]
    got = FHE.run_batch(batch)
    wrong = [i for i in range(BIG_BATCH) if got[i] != want[i % len(base)]]
    assert not wrong, [(i, got[i][0]) for i in wrong[:8]]
    structured = writer == "structured"
    for j in range(0, len(base), 17):
        if meta[j] is None:
            continue
        kind, ca, cb, rk = meta[j]
        assert want[j][1] == F.make_ciphertext(kind, bfv.mul_relin(ca, cb, rk)).to_bytes(structured=structured), j


def test_big_tiles_past_the_key_cache(keys, writer, tmp_path):
    """The same 2,112 calls in a fresh process whose key cache holds 4 keys (FHE_B200_KEY_CACHE=4): the tiles in flight pin
    their ~230 keys each past the capacity, keys are evicted between tiles and parsed again, and a churn of 64 other users
    in between evicts them once more.  Both runs equal the same calls in 16-call batches, byte for byte."""
    import hashlib
    import json

    from fhe_precompiles_b200 import FHE

    base, _ = big_batch(keys, user_keys(256))
    want = []
    for lo in range(0, len(base), 16):
        want += FHE.run_batch(base[lo: lo + 16])
    want = [[st, hashlib.sha256(out).hexdigest()] for st, out in want]
    out = tmp_path / "small_cache.json"
    env = dict(os.environ, FHE_B200_KEY_CACHE="4", FHE_B200_ZSTD_WRITER="1" if writer == "structured" else "0")
    r = subprocess.run([sys.executable, "-c", SMALL_CACHE, ROOT, str(out)], capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    got = json.loads(out.read_text())
    for run in ("first", "second"):
        wrong = [i for i in range(BIG_BATCH) if got[run][i] != want[i % len(base)]]
        assert not wrong, (run, [(i, got[run][i][0]) for i in wrong[:8]])


# ---------------------------------------------------------------- 4. launches
LAUNCHES = r"""
import sys
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
from helpers import KeySet, encrypt_value
from oracle import formats as F
from user_keys import user_keys
from fhe_precompiles_b200 import FHE, _lib, pack

keys = KeySet.load()
users = user_keys(256)
L = _lib.lib()
a = F.make_ciphertext("i64", encrypt_value(keys, "i64", 6, 8)).to_bytes()
b = F.make_ciphertext("i64", encrypt_value(keys, "i64", 7, 9)).to_bytes()
packed = [pack.pack_binary_operation(pub, a, b) for pub, _ in users]

def launches(name, n, n_keys):
    batch = [(name, packed[i % n_keys]) for i in range(n)]
    before = L.fhe_b200_launch_count()
    res = FHE.run_batch(batch, host_threads=1)
    assert all(st == 0 for st, _ in res)
    return L.fhe_b200_launch_count() - before

for n, keys_many in ((16, 16), (1024, 256)):
    for n_keys in (1, keys_many):  # every key parsed and on the device before the counted runs
        launches("mul_cipheri64_cipheri64", n, n_keys)
    print(n, launches("add_cipheri64_cipheri64", n, 1), launches("mul_cipheri64_cipheri64", n, 1),
          launches("mul_cipheri64_cipheri64", n, keys_many))
"""


def sequence_launches(dev):
    """(split, fused, prepare): the kernels of one multiply + relinearise below and at FUSED_TAIL_MIN_OPS ops, and of one group of
    prepared keys, counted on the device API (mul_relin_keyed adds one launch, its key table).  At 96 ops a group holds
    15 * 96 / 24 = 60 keys, so 61 keys take two groups."""
    import torch

    rng = np.random.default_rng(61)
    n = FUSED_TAIL_MIN_OPS
    a = to_dev(random_ct(rng, n))
    rks = to_dev(random_keys(rng, 61))

    def count(fn):
        before = dev.launch_count()
        fn()
        torch.cuda.synchronize()
        return dev.launch_count() - before

    split = count(lambda: dev.mul_relin(a[:1], a[:1], rks[0]))
    fused = count(lambda: dev.mul_relin(a, a, rks[0]))
    one = count(lambda: dev.mul_relin_keyed(a, a, rks[:1], torch.zeros(n, dtype=torch.int32).cuda()))
    two = count(lambda: dev.mul_relin_keyed(a, a, rks, torch.arange(n, dtype=torch.int32).cuda() % 61))
    assert one == fused + 1, (one, fused)
    return split, fused, two - one


def test_launches_of_multi_user_tiles(dev, writer):
    """One 16-call tile of ct-ct multiplies under 16 keys launches what the same tile under one key launches: the codec kernels
    and one split-tail sequence, not 16.  One 1,024-call tile under 256 keys launches the codec kernels and one fused sequence
    (the 256 keys prepared in one group: 15 * 1024 / 24 = 640 fit the tensor region), as under one key.  The codec launches are
    those of the same tile of additions, which runs one kernel."""
    split, fused, prepare = sequence_launches(dev)
    assert split > 0 and fused > 0 and prepare > 0, (split, fused, prepare)
    env = dict(os.environ, FHE_B200_TILE_OPS="1024", FHE_B200_ZSTD_WRITER="1" if writer == "structured" else "0")
    r = subprocess.run([sys.executable, "-c", LAUNCHES, ROOT], capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    rows = {int(l.split()[0]): [int(x) for x in l.split()[1:]] for l in r.stdout.splitlines() if l and l.split()[0].isdigit()}
    add16, mul16, mul16k = rows[16]
    assert mul16 == add16 - 1 + split, rows
    assert mul16k == mul16, rows
    add1k, mul1k, mul1kk = rows[1024]
    groups = -(-256 // (15 * 1024 // 24))
    assert mul1k == add1k - 1 + fused, rows
    assert mul1kk == mul1k + prepare * (groups - 1), rows


# ---------------------------------------------------------------- 5. real keys
def test_real_keys_round_trip(keys, writer):
    """One batch of multiplies under the tests/data key and the network key: each result, decrypted with its own secret key,
    is the product of the values"""
    from fhe_precompiles_b200 import FHE, pack

    calls, want = [], []
    for i in range(12):
        net = i % 2 == 1
        pub = keys.net_pub_bytes if net else keys.pub_bytes
        x, y = 3 + i, -(5 + 2 * i)
        ca = F.make_ciphertext("i64", encrypt_value(keys, "i64", x, 50 + i, network=net)).to_bytes()
        cb = F.make_ciphertext("i64", encrypt_value(keys, "i64", y, 80 + i, network=net)).to_bytes(structured=i % 3 == 0)
        calls.append(("mul_cipheri64_cipheri64", pack.pack_binary_operation(pub, ca, cb)))
        want.append((net, x * y))
    res = FHE.run_batch(calls)
    for (st, out), (net, prod) in zip(res, want):
        assert st == 0
        assert decrypt_value(keys, "i64", F.Ciphertext.from_bytes(out).polys(), network=net) == prod
