"""Device-resident batched entry points (part 2 of include/fhe_precompiles_b200.h) on torch CUDA tensors.

torch is plumbing only: it owns device memory and streams; every op is a call into the C-ABI library.
Tensors are int64 views of uint64 words (torch has no general uint64 ops), C-contiguous:
  ciphertext [n, 2, 2, 4096], size-3 ciphertext [n, 3, 2, 4096], relin key [2, 2, 3, 4096],
  plaintext [n, 4096] int16 (coefficients < 4096).
Typed values (encode / decode, encrypt_values / decrypt_values): u64 and i64 int64 [n] (u64 as its two's-complement view),
u256 int64 [n, 4] (words least significant first), frac64 float64 [n].
"""
from __future__ import annotations

import ctypes
from typing import Sequence

import torch

from . import _lib

N = 4096


def _check(rc: int) -> None:
    if rc != 0:
        raise RuntimeError("fhe_precompiles_b200: " + _lib.last_error())


def _dev(t: torch.Tensor) -> int:
    if not t.is_cuda:
        raise RuntimeError("fhe_precompiles_b200 has no CPU path: tensors must live on a CUDA device")
    if not t.is_contiguous():
        raise ValueError("tensor must be contiguous")
    return t.device.index if t.device.index is not None else torch.cuda.current_device()


def _stream(dev: int) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def init(device: int = 0) -> None:
    _check(_lib.lib().fhe_b200_init(device))


def launch_count() -> int:
    return int(_lib.lib().fhe_b200_launch_count())


def _binary(fn, a: torch.Tensor, b: torch.Tensor, out_shape) -> torch.Tensor:
    dev = _dev(a)
    _dev(b)
    n = a.shape[0]
    out = torch.empty(out_shape, dtype=torch.int64, device=a.device)
    _check(fn(dev, a.data_ptr(), b.data_ptr(), out.data_ptr(), n, _stream(dev)))
    return out


def add(a, b):
    return _binary(_lib.lib().fhe_b200_add, a, b, a.shape)


def sub(a, b):
    return _binary(_lib.lib().fhe_b200_sub, a, b, a.shape)


def negate(a):
    dev = _dev(a)
    out = torch.empty_like(a)
    _check(_lib.lib().fhe_b200_negate(dev, a.data_ptr(), out.data_ptr(), a.shape[0], _stream(dev)))
    return out


def plain_addsub(ct, plain, mode: int):
    dev = _dev(ct)
    _dev(plain)
    assert plain.dtype == torch.int16 and plain.shape == (ct.shape[0], N)
    out = torch.empty_like(ct)
    _check(_lib.lib().fhe_b200_plain_addsub(dev, ct.data_ptr(), plain.data_ptr(), out.data_ptr(), ct.shape[0], mode, _stream(dev)))
    return out


def multiply_plain(ct, plain):
    dev = _dev(ct)
    _dev(plain)
    assert plain.dtype == torch.int16 and plain.shape == (ct.shape[0], N)
    out = torch.empty_like(ct)
    _check(_lib.lib().fhe_b200_multiply_plain(dev, ct.data_ptr(), plain.data_ptr(), out.data_ptr(), ct.shape[0], _stream(dev)))
    return out


def multiply(a, b):
    return _binary(_lib.lib().fhe_b200_multiply, a, b, (a.shape[0], 3, 2, N))


def relinearize(c3, rk):
    return _binary(_lib.lib().fhe_b200_relinearize, c3, rk, (c3.shape[0], 2, 2, N))


def mul_relin(a, b, rk, out=None):
    dev = _dev(a)
    _dev(b)
    _dev(rk)
    if out is None:
        out = torch.empty_like(a)
    _check(_lib.lib().fhe_b200_mul_relin(dev, a.data_ptr(), b.data_ptr(), rk.data_ptr(), out.data_ptr(), a.shape[0], _stream(dev)))
    return out


def ntt_(data: torch.Tensor, mods: Sequence[int], inverse: bool = False) -> torch.Tensor:
    """In-place batched NTT over data[..., 4096]; limb i (flattened) uses modulus mods[i % len(mods)]."""
    dev = _dev(data)
    arr = (ctypes.c_int32 * len(mods))(*mods)
    _check(_lib.lib().fhe_b200_ntt(dev, data.data_ptr(), data.numel() // N, arr, len(mods), int(inverse), _stream(dev)))
    return data


def behz_extend(a, b):
    return _binary(_lib.lib().fhe_b200_behz_extend, a, b, (a.shape[0], 4, 5, N))


def behz_tensor(a, b):
    return _binary(_lib.lib().fhe_b200_behz_tensor, a, b, (a.shape[0], 3, 5, N))


def behz_floor_sk(tens):
    dev = _dev(tens)
    out = torch.empty((tens.shape[0], 3, 2, N), dtype=torch.int64, device=tens.device)
    _check(_lib.lib().fhe_b200_behz_floor_sk(dev, tens.data_ptr(), out.data_ptr(), tens.shape[0], _stream(dev)))
    return out


def mul_relin_host(a: torch.Tensor, b: torch.Tensor, rk: torch.Tensor, out: torch.Tensor, device: int = 0) -> torch.Tensor:
    """a, b, out: HOST tensors [n,2,2,4096] int64 (pinned for full PCIe rate); rk: host [2,2,3,4096]."""
    for t in (a, b, rk, out):
        if t.is_cuda or not t.is_contiguous():
            raise ValueError("mul_relin_host takes contiguous host tensors")
    _check(_lib.lib().fhe_b200_mul_relin_host(device, a.data_ptr(), b.data_ptr(), rk.data_ptr(), out.data_ptr(), a.shape[0]))
    return out


def mul_relin_frames(fa: torch.Tensor, fb: torch.Tensor, rk: torch.Tensor, out: torch.Tensor, status: torch.Tensor, device: int = 0) -> torch.Tensor:
    """fa, fb: HOST uint8 tensors [n, stride] whose rows start with a structured frame (stride >= frame_bytes()); out: host uint8
    [n, frame_stride()]; status: host int32 [n]; rk: host words [2,2,3,4096]."""
    for t in (fa, fb, rk, out, status):
        if t.is_cuda or not t.is_contiguous():
            raise ValueError("mul_relin_frames takes contiguous host tensors")
    if fa.shape != fb.shape or out.shape[1] != frame_stride() or status.numel() != fa.shape[0]:
        raise ValueError("mul_relin_frames: shape mismatch")
    _check(_lib.lib().fhe_b200_mul_relin_frames(device, fa.data_ptr(), fb.data_ptr(), fa.shape[1], rk.data_ptr(), out.data_ptr(), fa.shape[0],
                                                status.data_ptr()))
    return out


def upload_frames(frames: torch.Tensor, device: int = 0):
    """frames: HOST uint8 [n, stride] whose rows start with a structured frame -> (ct [n,2,2,4096] int64 on `device`, status [n] int32
    host: 0 ok, 1 rejected).  The serialized -> device-resident end of a chain of device-resident operations."""
    if frames.is_cuda or not frames.is_contiguous() or frames.dtype != torch.uint8:
        raise ValueError("upload_frames takes a contiguous host uint8 tensor")
    n = frames.shape[0]
    ct = torch.empty((n, 2, 2, N), dtype=torch.int64, device=torch.device("cuda", device))
    status = torch.zeros((n,), dtype=torch.int32)
    _check(_lib.lib().fhe_b200_upload_frames(device, frames.data_ptr(), frames.shape[1], n, ct.data_ptr(), status.data_ptr()))
    return ct, status


def download_frames(ct: torch.Tensor, out: torch.Tensor = None):
    """ct [n,2,2,4096] on a CUDA device -> (frames HOST uint8 [n, frame_stride()], status [n] int32: 0 ok, 2 constant ciphertext)."""
    dev = _dev(ct)
    n = ct.shape[0]
    torch.cuda.current_stream(dev).synchronize()  # the library copies on its own streams: ct must be complete
    if out is None:
        out = torch.zeros((n, frame_stride()), dtype=torch.uint8).pin_memory()
    status = torch.zeros((n,), dtype=torch.int32)
    _check(_lib.lib().fhe_b200_download_frames(dev, ct.data_ptr(), n, out.data_ptr(), status.data_ptr()))
    return out, status


def frame_bytes() -> int:
    return int(_lib.lib().fhe_b200_frame_bytes())


def frame_stride() -> int:
    return int(_lib.lib().fhe_b200_frame_stride())


KERNEL_NAMES = ("k_behz_tensor", "k_floor_sk", "k_relin_ks", "k_relin_finish", "k_ext_ntt", "k_tensor_intt", "k_digit_ntt", "k_ks_intt",
                "k_ext_conv", "k_ks_finish", "k_rk_prepare_ksd", "k_digit_ntt_ksd", "k_ks_intt_ksd", "k_ks_finish_ksd", "k_tensor_floor_d", "k_ks_tail_ksd")


def set_kernel_timing(on: bool) -> None:
    _lib.lib().fhe_b200_set_kernel_timing(int(on))


def kernel_timing_report(device: int = 0) -> dict:
    """{kernel: (total ms, launches)} accumulated by mul_relin() since the last report."""
    ms = (ctypes.c_double * len(KERNEL_NAMES))()
    cnt = (ctypes.c_uint64 * len(KERNEL_NAMES))()
    _check(_lib.lib().fhe_b200_kernel_timing_report(device, ms, cnt))
    return {KERNEL_NAMES[i]: (float(ms[i]), int(cnt[i])) for i in range(len(KERNEL_NAMES)) if cnt[i]}


def parse_public_key(data: bytes):
    """PublicKey bytes -> (pk [2,3,4096], rk [2,2,3,4096]) int64 host tensors, via the library's codec."""
    pk = torch.empty((2, 3, N), dtype=torch.int64)
    rk = torch.empty((2, 2, 3, N), dtype=torch.int64)
    rc = _lib.lib().fhe_b200_parse_public_key(data, len(data), pk.data_ptr(), rk.data_ptr())
    if rc != 0:
        raise RuntimeError(f"parse_public_key failed with code {rc}")
    return pk, rk


def int_peak(device: int = 0, wide=True) -> float:
    """Measured integer multiply-add peak in 1e12 mad/s (mad.wide.u32 or mad.lo.u32 microbenchmark)."""
    v = ctypes.c_double()
    _check(_lib.lib().fhe_b200_int_peak(device, int(wide), ctypes.byref(v)))
    return float(v.value)


def bfly_peak(device: int = 0, mod: int = 0) -> float:
    """Register-only NTT butterfly rate in 1e9 butterflies/s (mod 0-2: small primes, 3-5: 61-bit primes)."""
    v = ctypes.c_double()
    _check(_lib.lib().fhe_b200_bfly_peak(device, mod, ctypes.byref(v)))
    return float(v.value)


def set_fused(on: bool) -> None:
    """Select the multi-polynomial-per-CTA kernels (True) or the one-polynomial-per-CTA kernels (False, default)."""
    _lib.lib().fhe_b200_set_fused(int(on))


def encrypt(pk: torch.Tensor, plain: torch.Tensor, seeds: torch.Tensor) -> torch.Tensor:
    """pk [2,3,4096] int64, plain [n,4096] int16, seeds [n,8] int64 -- one 512-bit seed per op -- (all on one CUDA device)
    -> ct [n,2,2,4096]."""
    dev = _dev(pk)
    _dev(plain)
    _dev(seeds)
    n = plain.shape[0]
    assert plain.dtype == torch.int16 and seeds.dtype == torch.int64 and tuple(seeds.shape) == (n, 8)
    ct = torch.empty((n, 2, 2, N), dtype=torch.int64, device=pk.device)
    _check(_lib.lib().fhe_b200_encrypt(dev, pk.data_ptr(), plain.data_ptr(), seeds.data_ptr(), ct.data_ptr(), n, _stream(dev)))
    return ct


def seal_sample(draws: torch.Tensor):
    """draws [n, 28672] int32 on a CUDA device (32-bit draws in stream order) -> (u, e0, e1 as int8 [n, 4096] each, failed
    int32 [n]): SEAL's sample_poly_ternary + 2 x sample_poly_normal on those draws (the sampling stage of encrypt())."""
    dev = _dev(draws)
    n = draws.shape[0]
    words = int(_lib.lib().fhe_b200_seal_op_words())
    assert draws.dtype == torch.int32 and draws.shape[1] == 28 * 1024
    buf = torch.zeros((n, words), dtype=torch.int64, device=draws.device)
    buf[:, : 28 * 512] = draws.contiguous().view(torch.int64)
    failed = torch.zeros(n, dtype=torch.int32, device=draws.device)
    _check(_lib.lib().fhe_b200_seal_sample(dev, buf.data_ptr(), failed.data_ptr(), n, _stream(dev)))
    smp = buf[:, 28 * 512 :].contiguous().view(torch.int8).reshape(n, 3, N)
    return smp[:, 0], smp[:, 1], smp[:, 2], failed


def decrypt(ct: torch.Tensor, sk: torch.Tensor) -> torch.Tensor:
    """ct [n,2,2,4096], sk [>=2,4096] int64 (NTT form) -> plaintext coefficients [n,4096] int16."""
    dev = _dev(ct)
    _dev(sk)
    plain = torch.empty((ct.shape[0], N), dtype=torch.int16, device=ct.device)
    _check(_lib.lib().fhe_b200_decrypt(dev, ct.data_ptr(), sk.data_ptr(), plain.data_ptr(), ct.shape[0], _stream(dev)))
    return plain


def decrypt_checked(ct: torch.Tensor, sk: torch.Tensor):
    """decrypt() plus SEAL's invariant-noise-budget test: returns (plain [n,4096] int16, exhausted [n] int32), exhausted[i] = 1
    where ciphertext i has no noise budget left (its plaintext is meaningless; the byte surface returns code 5 there)."""
    dev = _dev(ct)
    _dev(sk)
    plain = torch.empty((ct.shape[0], N), dtype=torch.int16, device=ct.device)
    flags = torch.empty((ct.shape[0],), dtype=torch.int32, device=ct.device)
    _check(_lib.lib().fhe_b200_decrypt_checked(dev, ct.data_ptr(), sk.data_ptr(), plain.data_ptr(), flags.data_ptr(), ct.shape[0], _stream(dev)))
    return plain, flags


# value kinds, numbered as fhe_b200_data_type_kind numbers them
VALUE_KINDS = ("u256", "u64", "i64", "frac64")


def _value_kind(kind: str) -> int:
    if kind not in VALUE_KINDS:
        raise ValueError(f"unknown value kind {kind!r}: expected one of {', '.join(VALUE_KINDS)}")
    return VALUE_KINDS.index(kind)


def _value_shape(kind: str, n: int):
    return (n, 4) if kind == "u256" else (n,)


def _value_dtype(kind: str):
    return torch.float64 if kind == "frac64" else torch.int64


def encode(kind: str, values: torch.Tensor):
    """values ([n] int64 for u64 / i64, [n, 4] int64 for u256, [n] float64 for frac64) -> (plain [n, 4096] int16, status [n]
    int32): sunscreen's plaintext of each value, bit-identical to the byte surface's encoder.  status[i] = 7 (and a zero row)
    where a frac64 value is NaN, +-inf or |v| >= 2^64, 0 otherwise."""
    k = _value_kind(kind)
    dev = _dev(values)
    n = values.shape[0]
    if values.dtype != _value_dtype(kind) or tuple(values.shape) != _value_shape(kind, n):
        raise ValueError(f"encode({kind!r}): values must be {_value_dtype(kind)} {_value_shape(kind, 'n')}")
    plain = torch.empty((n, N), dtype=torch.int16, device=values.device)
    status = torch.empty((n,), dtype=torch.int32, device=values.device)
    _check(_lib.lib().fhe_b200_encode_values(dev, k, values.data_ptr(), plain.data_ptr(), status.data_ptr(), n, _stream(dev)))
    return plain, status


def decode(kind: str, plain: torch.Tensor) -> torch.Tensor:
    """plain [n, 4096] int16 -> values in encode()'s layout: the byte surface's decoder applied to every row, whatever its
    coefficients (>= 4096 wrap as the reference's do)."""
    k = _value_kind(kind)
    dev = _dev(plain)
    if plain.dtype != torch.int16 or plain.dim() != 2 or plain.shape[1] != N:
        raise ValueError("decode: plain must be int16 [n, 4096]")
    n = plain.shape[0]
    values = torch.empty(_value_shape(kind, n), dtype=_value_dtype(kind), device=plain.device)
    _check(_lib.lib().fhe_b200_decode_values(dev, k, plain.data_ptr(), values.data_ptr(), n, _stream(dev)))
    return values


def encrypt_values(pk: torch.Tensor, kind: str, values: torch.Tensor, seeds: torch.Tensor):
    """encode() + encrypt(): (ct [n,2,2,4096], status [n] int32 as encode() returns it)."""
    plain, status = encode(kind, values)
    return encrypt(pk, plain, seeds), status


def decrypt_values(ct: torch.Tensor, sk: torch.Tensor, kind: str):
    """decrypt_checked() + decode(): (values, exhausted [n] int32); values[i] is meaningless where exhausted[i] = 1."""
    plain, exhausted = decrypt_checked(ct, sk)
    return decode(kind, plain), exhausted


def set_chunk_ops(ops: int) -> int:
    """Ops per chunk of the device-resident entry points (default 4,096); ops <= 0 only queries. Returns the previous value."""
    prev = int(_lib.lib().fhe_b200_set_chunk_ops(int(ops)))
    if prev < 0:
        raise RuntimeError("fhe_precompiles_b200: " + _lib.last_error())
    return prev
