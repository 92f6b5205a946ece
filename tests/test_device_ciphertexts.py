"""Device-resident chains from and to sunscreen Ciphertext bytes: fhe_b200_upload_ciphertexts / fhe_b200_download_ciphertexts and
device.upload_ciphertexts / download_ciphertexts, compared byte for byte with the c_fhe_* precompiles on the same ciphertexts,
under both result writers, and status for status with c_fhe_add_cipherK_cipherK on every operand form and every rejection.
Run on the B200 box: pytest -m gpu."""
import ctypes
import os
import struct
import subprocess
import sys
import zlib

import numpy as np
import pytest

from helpers import KINDS, MODULI, N, ROOT, random_ct
from oracle import formats as F

pytestmark = pytest.mark.gpu

PUBLIC = bytes([4, 5, 6])


@pytest.fixture(scope="module")
def dev():
    import torch

    from fhe_precompiles_b200 import device

    assert torch.cuda.is_available(), "no CUDA device: the product has no CPU path"
    device.init(0)
    return device


@pytest.fixture(scope="module")
def L():
    from fhe_precompiles_b200 import _lib

    return _lib.lib()


class Writer:
    """fhe_b200_set_zstd_writer(mode) for the duration of a with-block, restored afterwards"""

    def __init__(self, L, mode: int):
        self.L, self.mode = L, mode

    def __enter__(self):
        self.prev = self.L.fhe_b200_set_zstd_writer(self.mode)

    def __exit__(self, *exc):
        self.L.fhe_b200_set_zstd_writer(self.prev)


def to_dev(a: np.ndarray):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()


def to_np(t) -> np.ndarray:
    return t.cpu().numpy().view(np.uint64)


def small_values(kind: str, n: int, seed: int) -> list:
    rng = np.random.default_rng(seed)
    vals = [int(v) for v in rng.integers(0, 1000, n)]
    return [float(v) / 4 for v in vals] if kind == "frac64" else vals


def encrypt_all(L, kind: str, vals, mode: int) -> list:
    """c_fhe_encrypt_<kind> of every value (network key) under writer `mode`"""
    from fhe_precompiles_b200 import FHE, pack

    with Writer(L, mode):
        return [getattr(FHE, f"encrypt_{kind}")(pack.pack_two_arguments(pack.SERIALIZE[kind](v), PUBLIC)) for v in vals]


def three(kind: str, n: int):
    """the plaintext of 3 (3.0 for frac64) n times, encoded on the device"""
    import torch

    if kind == "frac64":
        return torch.full((n,), 3.0, dtype=torch.float64).cuda()
    if kind == "u256":
        t = torch.zeros((n, 4), dtype=torch.int64)
        t[:, 0] = 3
        return t.cuda()
    return torch.full((n,), 3, dtype=torch.int64).cuda()


def parse_words(L, ct: bytes):
    """fhe_b200_parse_ciphertext: (code, words [2][2][N])"""
    words = np.zeros((2, 2, N), dtype=np.uint64)
    rc = L.fhe_b200_parse_ciphertext(ct, len(ct), words.ctypes.data, None, 0)
    return rc, words


def add_code(keys, kind: str, a: bytes, b: bytes) -> int:
    """the code c_fhe_add_cipher<kind>_cipher<kind>(pack(pk, a, b)) returns"""
    from fhe_precompiles_b200 import FHE, FheError, pack

    try:
        getattr(FHE, f"add_cipher{kind}_cipher{kind}")(pack.pack_binary_operation(keys.net_pub_bytes, a, b))
        return 0
    except FheError as e:
        return e.code


def ciphertext_bytes(kind: str, blob: bytes) -> bytes:
    """bincode(sunscreen::Ciphertext) of `kind` around an arbitrary SEAL blob"""
    dt = F.data_type_string(kind).encode()
    return struct.pack("<Q", len(dt)) + dt + struct.pack("<IQ", 0, 1) + F.WithContext(F.Params(), blob).to_bytes()


@pytest.mark.parametrize("mode", [0, 1], ids=["seal", "structured"])
@pytest.mark.parametrize("kind", KINDS)
def test_chain_matches_the_precompiles(dev, keys, L, kind, mode):
    """download(op(upload(A), upload(B)), kind) equals c_fhe_<op>(pack(pk, A, B)) byte for byte, A and B being c_fhe_encrypt_<kind>
    outputs in SEAL's bytes: multiply + relinearise, add, sub, and two plaintext ops after encode, under both writers."""
    from fhe_precompiles_b200 import FHE, pack

    n = 4
    A = encrypt_all(L, kind, small_values(kind, n, 1), 0)
    B = encrypt_all(L, kind, small_values(kind, n, 2), 0)
    ser3 = pack.SERIALIZE[kind](3.0 if kind == "frac64" else 3)
    with Writer(L, mode):
        da, sa = dev.upload_ciphertexts(A, kind)
        db, sb = dev.upload_ciphertexts(B, kind)
        assert sa.tolist() == [0] * n and sb.tolist() == [0] * n
        plain, pst = dev.encode(kind, three(kind, n))
        assert not pst.cpu().numpy().any()
        chains = {
            f"mul_cipher{kind}_cipher{kind}": (dev.mul_relin(da, db, to_dev(keys.net_rk)), B),
            f"add_cipher{kind}_cipher{kind}": (dev.add(da, db), B),
            f"sub_cipher{kind}_cipher{kind}": (dev.sub(da, db), B),
            f"mul_cipher{kind}_{kind}": (dev.multiply_plain(da, plain), [ser3] * n),
            f"add_cipher{kind}_{kind}": (dev.plain_addsub(da, plain, 0), [ser3] * n),
        }
        for name, (res, second) in chains.items():
            got, st = dev.download_ciphertexts(res, kind)
            assert st.tolist() == [0] * n, name
            for i in range(n):
                want = getattr(FHE, name)(pack.pack_binary_operation(keys.net_pub_bytes, A[i], second[i]))
                assert got[i] == want, f"{name} [{i}]"


@pytest.mark.parametrize("kind", KINDS)
def test_round_trip(dev, L, kind):
    """download(upload(X)) == X for default-writer outputs, and for structured-writer outputs downloaded under that writer"""
    for mode in (0, 1):
        X = encrypt_all(L, kind, small_values(kind, 3, 7 + mode), mode)
        with Writer(L, mode):
            d, st = dev.upload_ciphertexts(X, kind)
            assert st.tolist() == [0, 0, 0]
            back, st2 = dev.download_ciphertexts(d, kind)
        assert st2.tolist() == [0, 0, 0] and back == X, f"writer {mode}"


def mixed_batch(kind: str, n: int):
    """n ciphertexts of `kind` in every operand form, mostly SEAL's libzstd frames (the device decoder's threshold is met in the
    first chunk), with every kind of rejection among the first 127 rows; returns (cts, {row: what})"""
    rng = np.random.default_rng(97)
    polys = random_ct(rng, n)
    other = "frac64" if kind != "frac64" else "i64"  # (u64 and u256 share sunscreen's Unsigned data_type)
    cts = [F.make_ciphertext(kind, p).to_bytes() for p in polys]
    forms = {}
    for i in list(range(5, n, 37)) + [n - 1]:
        cts[i] = F.make_ciphertext(kind, polys[i]).to_bytes(structured=True)
        forms[i] = "structured"
    for i in range(11, n, 41):
        cts[i] = F.make_ciphertext(kind, polys[i]).to_bytes(compr=F.COMPR_NONE)
        forms[i] = "compr none"
    for i in range(13, n, 43):
        cts[i] = F.make_ciphertext(kind, polys[i]).to_bytes(compr=F.COMPR_ZLIB)
        forms[i] = "zlib"
    bad = dict.fromkeys(range(20, 30))
    good = cts[0]
    cts[20] = good[:7] + b"\x01" + good[8:]  # data_type length beyond the buffer: bad framing
    cts[21] = good[:-7]  # truncated bincode
    cts[22] = F.make_ciphertext(other, polys[22]).to_bytes()  # wrong data_type
    size3 = np.concatenate([polys[23], polys[23][:1]])
    cts[23] = F.make_ciphertext(kind, size3).to_bytes()  # a size-3 ciphertext
    over = polys[24].copy()
    over[1, 1, N - 1] = MODULI[1]
    cts[24] = F.make_ciphertext(kind, over).to_bytes()  # residue >= q, libzstd
    cts[25] = F.make_ciphertext(kind, over).to_bytes(structured=True)  # residue >= q, structured frame
    frame = F.zstd().compress(F.fresh_data_ciphertext(polys[26]).payload(), 3)
    cut = frame[: len(frame) // 2]
    cts[26] = ciphertext_bytes(kind, F.seal_header(F.COMPR_ZSTD, 16 + len(cut)) + cut)  # truncated frame
    zl = zlib.compress(F.fresh_data_ciphertext(polys[27]).payload())[:-9]
    cts[27] = ciphertext_bytes(kind, F.seal_header(F.COMPR_ZLIB, 16 + len(zl)) + zl)  # truncated zlib stream
    cts[28] = ciphertext_bytes(kind, F.seal_header(F.COMPR_NONE, 16 + 100) + bytes(100))  # uncompressed, wrong size
    cts[29] = ciphertext_bytes(kind, b"\x00" * 16 + frame)  # not a SEAL header
    forms.update(bad)
    return cts, forms


@pytest.mark.parametrize("kind", ["i64", "u256"])
def test_every_operand_form_in_one_batch(dev, keys, L, kind):
    """300 ciphertexts (two chunks): SEAL libzstd, structured, compr_mode none and zlib blobs, bad framing, a wrong data_type, a
    size-3 ciphertext, residues >= q, truncated frames.  Every status equals c_fhe_add_cipherK_cipherK's code with that row as
    first operand, accepted rows hold fhe_b200_parse_ciphertext's words, and the device decoder ran.  The same rows at n = 127
    and n = 1 (host inflate) give the same statuses."""
    n = 300
    cts, forms = mixed_batch(kind, n)
    good = cts[0]
    want = [add_code(keys, kind, c, good) for c in cts]
    assert [i for i in range(n) if want[i]] == list(range(20, 30)), want[:40]
    before = dev.launch_count()
    d, st = dev.upload_ciphertexts(cts, kind)
    launches = dev.launch_count() - before
    assert st.tolist() == want
    assert launches >= 4 + 2, f"{launches} launches: the device zstd decoder did not run"
    words = to_np(d)
    for i in range(n):
        if want[i] == 0:
            rc, w = parse_words(L, cts[i])
            assert rc == 0 and np.array_equal(words[i], w), f"row {i} ({forms.get(i, 'libzstd')})"
    before = dev.launch_count()
    d127, st127 = dev.upload_ciphertexts(cts[:127], kind)
    assert dev.launch_count() - before <= 2  # payloads and structured frames only: the host inflated
    assert st127.tolist() == want[:127]
    assert np.array_equal(to_np(d127)[[i for i in range(127) if want[i] == 0]], words[[i for i in range(127) if want[i] == 0]])
    for i in sorted(set(forms) | {0, 1}):
        if i < 127:
            d1, st1 = dev.upload_ciphertexts([cts[i]], kind)
            assert st1.tolist() == [want[i]], f"row {i} alone"
            if want[i] == 0:
                assert np.array_equal(to_np(d1)[0], words[i])


@pytest.mark.parametrize("mode", [0, 1], ids=["seal", "structured"])
def test_transparent_result(dev, keys, L, mode):
    """a constant (transparent) result downloads to the byte surface's bytes for it"""
    from fhe_precompiles_b200 import FHE, pack

    kind = "u64"
    A = encrypt_all(L, kind, [5, 9], 0)
    with Writer(L, mode):
        d, _ = dev.upload_ciphertexts(A, kind)
        got, st = dev.download_ciphertexts(dev.sub(d, d), kind)
        want = [FHE.sub_cipheru64_cipheru64(pack.pack_binary_operation(keys.net_pub_bytes, a, a)) for a in A]
    assert st.tolist() == [0, 0] and got == want


def test_empty_and_bad_arguments(dev, L):
    import torch

    d, st = dev.upload_ciphertexts([], "i64")
    assert tuple(d.shape) == (0, 2, 2, N) and st.numel() == 0
    out, st = dev.download_ciphertexts(torch.zeros((0, 2, 2, N), dtype=torch.int64).cuda(), "i64")
    assert out == [] and st.numel() == 0
    assert L.fhe_b200_upload_ciphertexts(0, 1, None, None, 0, None, None) == 0
    assert L.fhe_b200_download_ciphertexts(0, 1, None, 0, None, None, None) == 0
    ct = bytes(10)
    ptrs, lens = (ctypes.c_char_p * 1)(ct), (ctypes.c_size_t * 1)(len(ct))
    status = (ctypes.c_int32 * 1)()
    words = torch.zeros((1, 2, 2, N), dtype=torch.int64).cuda()
    assert L.fhe_b200_upload_ciphertexts(0, 9, ptrs, lens, 1, words.data_ptr(), status) == -1
    assert "unknown kind" in L.fhe_b200_last_error().decode()
    outs, olens = (ctypes.c_void_p * 1)(), (ctypes.c_int64 * 1)()
    assert L.fhe_b200_download_ciphertexts(0, -1, words.data_ptr(), 1, outs, olens, status) == -1
    assert "unknown kind" in L.fhe_b200_last_error().decode()
    with pytest.raises(ValueError):
        dev.upload_ciphertexts([ct], "u128")
    with pytest.raises(TypeError):
        dev.upload_ciphertexts(ct, "i64")


NO_DEVICE = r"""
import ctypes, sys
sys.path.insert(0, sys.argv[1])
from fhe_precompiles_b200 import _lib
L = _lib.lib()
ct = bytes(200)
ptrs, lens, status = (ctypes.c_char_p * 1)(ct), (ctypes.c_size_t * 1)(len(ct)), (ctypes.c_int32 * 1)()
words = (ctypes.c_uint64 * 16384)()
assert L.fhe_b200_upload_ciphertexts(0, 2, ptrs, lens, 1, words, status) == -1
assert L.fhe_b200_last_error()
outs, olens = (ctypes.c_void_p * 1)(), (ctypes.c_int64 * 1)()
assert L.fhe_b200_download_ciphertexts(0, 2, words, 1, outs, olens, status) == -1
assert L.fhe_b200_last_error()
print("ok")
"""


def test_no_device_is_an_error():
    """without a CUDA device both entry points fail (-1), they never compute on the CPU"""
    r = subprocess.run([sys.executable, "-c", NO_DEVICE, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr
