"""ctypes loader of libfhe_precompiles_b200.so (the C-ABI boundary, include/fhe_precompiles_b200.h).

The library is built in-tree by `__graft_entry__.build()` / `make -C fhe_precompiles_b200/csrc`.
There is no fallback: a missing library raises, and every compute entry point fails without a CUDA device.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfhe_precompiles_b200.so")

TYPES = ("u256", "u64", "i64", "frac64")
BINARY_OPS = tuple(
    name
    for t in TYPES
    for o in ("add", "sub", "mul")
    for name in (f"{o}_cipher{t}_cipher{t}", f"{o}_cipher{t}_{t}", f"{o}_{t}_cipher{t}")
)
THRESHOLD_OPS = tuple(f"{o}_{t}" for o in ("encrypt", "reencrypt", "decrypt") for t in TYPES) + ("public_key_bytes",)
PRECOMPILES = BINARY_OPS + THRESHOLD_OPS  # the 49 names stamped at c_fhe.rs:74-141

_lib = None


class BatchCall(ctypes.Structure):
    _fields_ = [
        ("op", ctypes.c_int32),
        ("status", ctypes.c_int32),
        ("bytes", ctypes.c_void_p),
        ("bytes_length", ctypes.c_size_t),
        ("output", ctypes.c_void_p),
        ("output_length", ctypes.c_int64),
    ]


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        # not a fallback: this compiles the same CUDA library in-tree (nvcc, sm_100a) when a checkout has no binary yet
        import subprocess

        try:
            subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), "-j", str(os.cpu_count() or 4)], check=True,
                           stdout=subprocess.DEVNULL)
        except Exception as e:  # noqa: BLE001
            raise RuntimeError(
                f"{LIB_PATH} is missing and could not be built ({e}); build it with "
                "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). There is no CPU fallback."
            ) from e
    L = ctypes.CDLL(LIB_PATH)
    vp, sz, i32, i64 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int32, ctypes.c_int64
    for name in PRECOMPILES:
        fn = getattr(L, "c_fhe_" + name)
        fn.restype = i32
        fn.argtypes = [vp, sz, ctypes.POINTER(vp), ctypes.POINTER(i64)]
    L.fhe_free.argtypes = [vp]
    L.fhe_free.restype = None
    L.fhe_error.argtypes = [i32]
    L.fhe_error.restype = ctypes.c_char_p
    L.fhe_b200_last_error.restype = ctypes.c_char_p
    L.fhe_b200_device_count.restype = i32
    L.fhe_b200_init.argtypes = [i32]
    L.fhe_b200_init.restype = i32
    L.fhe_b200_launch_count.restype = ctypes.c_uint64
    L.fhe_b200_op_index.argtypes = [ctypes.c_char_p]
    L.fhe_b200_op_index.restype = i32
    L.fhe_b200_op_name.argtypes = [i32]
    L.fhe_b200_op_name.restype = ctypes.c_char_p
    L.fhe_b200_batch.argtypes = [ctypes.POINTER(BatchCall), sz, i32]
    L.fhe_b200_batch.restype = i64
    dev3 = [i32, vp, vp, vp, sz, vp]
    for name in ("add", "sub", "multiply", "relinearize"):
        getattr(L, "fhe_b200_" + name).argtypes = dev3
    L.fhe_b200_negate.argtypes = [i32, vp, vp, sz, vp]
    L.fhe_b200_plain_addsub.argtypes = [i32, vp, vp, vp, sz, i32, vp]
    L.fhe_b200_multiply_plain.argtypes = [i32, vp, vp, vp, sz, vp]
    L.fhe_b200_mul_relin.argtypes = [i32, vp, vp, vp, vp, sz, vp]
    L.fhe_b200_mul_relin_keyed.argtypes = [i32, vp, vp, vp, sz, vp, vp, sz, vp]
    L.fhe_b200_mul_relin_keyed.restype = i32
    L.fhe_b200_relinearize_keyed.argtypes = [i32, vp, vp, sz, vp, vp, sz, vp]
    L.fhe_b200_relinearize_keyed.restype = i32
    L.fhe_b200_encrypt.argtypes = [i32, vp, vp, vp, vp, sz, vp]
    L.fhe_b200_encrypt.restype = i32
    L.fhe_b200_encrypt_keyed.argtypes = [i32, vp, sz, vp, vp, vp, vp, sz, vp]
    L.fhe_b200_encrypt_keyed.restype = i32
    L.fhe_b200_seal_sample.argtypes = [i32, vp, vp, sz, vp]
    L.fhe_b200_seal_sample.restype = i32
    L.fhe_b200_seal_op_words.argtypes = []
    L.fhe_b200_seal_op_words.restype = sz
    L.fhe_b200_decrypt.argtypes = [i32, vp, vp, vp, sz, vp]
    L.fhe_b200_decrypt.restype = i32
    L.fhe_b200_decrypt_checked.argtypes = [i32, vp, vp, vp, vp, sz, vp]
    L.fhe_b200_decrypt_checked.restype = i32
    L.fhe_b200_encode_values.argtypes = [i32, i32, vp, vp, vp, sz, vp]
    L.fhe_b200_encode_values.restype = i32
    L.fhe_b200_decode_values.argtypes = [i32, i32, vp, vp, sz, vp]
    L.fhe_b200_decode_values.restype = i32
    L.fhe_b200_data_type_kind.argtypes = [ctypes.c_char_p]
    L.fhe_b200_data_type_kind.restype = i32
    L.fhe_b200_set_chunk_ops.argtypes = [i64]
    L.fhe_b200_set_chunk_ops.restype = i64
    L.fhe_b200_mul_relin_host.argtypes = [i32, vp, vp, vp, vp, sz]
    L.fhe_b200_mul_relin_host.restype = i32
    L.fhe_b200_mul_relin_frames.argtypes = [i32, vp, vp, sz, vp, vp, sz, vp]
    L.fhe_b200_mul_relin_frames.restype = i32
    L.fhe_b200_upload_frames.argtypes = [i32, vp, sz, sz, vp, vp]
    L.fhe_b200_upload_frames.restype = i32
    L.fhe_b200_download_frames.argtypes = [i32, vp, sz, vp, vp]
    L.fhe_b200_download_frames.restype = i32
    L.fhe_b200_upload_ciphertexts.argtypes = [i32, i32, vp, vp, sz, vp, vp]
    L.fhe_b200_upload_ciphertexts.restype = i32
    L.fhe_b200_download_ciphertexts.argtypes = [i32, i32, vp, sz, vp, vp, vp]
    L.fhe_b200_download_ciphertexts.restype = i32
    L.fhe_b200_frame_bytes.argtypes = []
    L.fhe_b200_frame_bytes.restype = sz
    L.fhe_b200_frame_stride.argtypes = []
    L.fhe_b200_frame_stride.restype = sz
    L.fhe_b200_int_peak.argtypes = [i32, i32, ctypes.POINTER(ctypes.c_double)]
    L.fhe_b200_int_peak.restype = i32
    L.fhe_b200_bfly_peak.argtypes = [i32, i32, ctypes.POINTER(ctypes.c_double)]
    L.fhe_b200_bfly_peak.restype = i32
    L.fhe_b200_set_call_timing.argtypes = [i32]
    L.fhe_b200_set_call_timing.restype = None
    L.fhe_b200_last_call_breakdown.argtypes = [ctypes.POINTER(ctypes.c_double)]
    L.fhe_b200_last_call_breakdown.restype = None
    L.fhe_b200_set_kernel_timing.argtypes = [i32]
    L.fhe_b200_set_kernel_timing.restype = None
    L.fhe_b200_kernel_timing_report.argtypes = [i32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint64)]
    L.fhe_b200_kernel_timing_report.restype = i32
    L.fhe_b200_ntt.argtypes = [i32, vp, sz, ctypes.POINTER(i32), i32, i32, vp]
    for name in ("add", "sub", "negate", "plain_addsub", "multiply_plain", "multiply", "relinearize", "mul_relin", "ntt"):
        getattr(L, "fhe_b200_" + name).restype = i32
    L.fhe_b200_parse_public_key.argtypes = [vp, sz, vp, vp]
    L.fhe_b200_parse_public_key.restype = i32
    L.fhe_b200_parse_private_key.argtypes = [vp, sz, vp]
    L.fhe_b200_parse_private_key.restype = i32
    L.fhe_b200_parse_ciphertext.argtypes = [vp, sz, vp, ctypes.c_char_p, sz]
    L.fhe_b200_parse_ciphertext.restype = i32
    L.fhe_b200_write_ciphertext.argtypes = [vp, ctypes.c_char_p, ctypes.POINTER(vp), ctypes.POINTER(i64)]
    L.fhe_b200_write_ciphertext.restype = i32
    L.fhe_b200_zstd_inflate.argtypes = [i32, vp, vp, ctypes.c_size_t, vp, vp, vp]
    L.fhe_b200_zstd_inflate.restype = i32
    L.fhe_b200_sha512.argtypes = [vp, ctypes.c_size_t, i32, vp]
    L.fhe_b200_sha512.restype = None
    L.fhe_b200_set_zstd_writer.argtypes = [i32]
    L.fhe_b200_set_zstd_writer.restype = i32
    L.fhe_b200_parms_id.argtypes = [i32, vp]
    L.fhe_b200_parms_id.restype = None
    _lib = L
    return L


def last_error() -> str:
    return lib().fhe_b200_last_error().decode(errors="replace")
