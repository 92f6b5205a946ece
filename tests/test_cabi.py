"""The C-ABI shared library loads and exports every symbol include/fhe_precompiles_b200.h declares; without a GPU
every compute entry point fails loudly (there is no CPU fallback).  CPU only."""
import ctypes
import os
import re

import pytest

from helpers import ROOT


@pytest.fixture(scope="module")
def lib():
    from fhe_precompiles_b200 import _lib

    return _lib.lib()


def declared_symbols():
    hdr = open(os.path.join(ROOT, "include/fhe_precompiles_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"FHE_PRECOMPILE\((\w+)\);", hdr))
    syms = {"c_fhe_" + n for n in names}
    syms |= set(re.findall(r"\b(fhe_b200_\w+|fhe_free|fhe_error)\s*\(", hdr))
    syms.discard("fhe_b200_call")
    return syms


def test_reference_surface_is_complete(lib):
    from fhe_precompiles_b200 import _lib

    # the 49 names of c_fhe.rs:74-141 + fhe_free + fhe_error
    assert len(_lib.PRECOMPILES) == 49 and len(set(_lib.PRECOMPILES)) == 49
    ref = open(os.path.join(ROOT, "tests/data/c_fhe_symbols.txt")).read().split()
    assert sorted(ref) == sorted(_lib.PRECOMPILES)
    for n in _lib.PRECOMPILES:
        assert hasattr(lib, "c_fhe_" + n)


def test_every_declared_symbol_is_exported(lib):
    syms = declared_symbols()
    assert len(syms) >= 51 + 20
    missing = [s for s in sorted(syms) if not hasattr(lib, s)]
    assert not missing, missing


def test_error_strings_match_lib_rs(lib):
    want = {1: "Unexpected end of file", 2: "Platform architecture invalid", 3: "Invalid encoding", 4: "Overflow in FHE program",
            5: "Invalid decryption", 6: "Invalid encryption", 7: "Base sunscreen error", 0: "Unknown error", 99: "Unknown error"}
    for code, msg in want.items():
        assert lib.fhe_error(code).decode() == msg


def test_op_table(lib):
    from fhe_precompiles_b200 import _lib

    for n in _lib.PRECOMPILES:
        idx = lib.fhe_b200_op_index(n.encode())
        assert idx >= 0 and lib.fhe_b200_op_name(idx).decode() == n
    assert lib.fhe_b200_op_index(b"nope") == -1


def test_public_key_bytes_needs_no_gpu(lib):
    from fhe_precompiles_b200 import FHE

    assert FHE.public_key_bytes() == open(os.path.join(ROOT, "fhe_precompiles_b200/data/network.pub"), "rb").read()


NO_DEVICE = r"""
import sys
sys.path.insert(0, sys.argv[1])
import pytest
import torch
assert not torch.cuda.is_available()
from fhe_precompiles_b200 import FHE, FheError, _lib

with pytest.raises(FheError) as e:
    FHE.add_cipheri64_cipheri64(b"\x00" * 16)
assert e.value.code == 7 and "no CPU fallback" in str(e.value)
assert _lib.lib().fhe_b200_init(0) == -1
from fhe_precompiles_b200 import device

with pytest.raises(RuntimeError):
    device.add(torch.zeros((1, 2, 2, 4096), dtype=torch.int64), torch.zeros((1, 2, 2, 4096), dtype=torch.int64))
print("ok")
"""


def test_no_cpu_fallback():
    """On a box without a CUDA device the product path must fail loudly, never compute on the CPU.  The check runs in a child
    process that sees no device (CUDA_VISIBLE_DEVICES empty), so it runs on GPU machines too."""
    import subprocess
    import sys

    r = subprocess.run([sys.executable, "-c", NO_DEVICE, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "fhe_precompiles_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cpp", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "import oracle" not in text and "from oracle" not in text and "bfv_oracle" not in text, f


def test_header_is_valid_c(tmp_path):
    """include/fhe_precompiles_b200.h must be consumable by a plain C compiler (cgo, JNI stubs ...)."""
    import subprocess

    src = tmp_path / "use.c"
    src.write_text('#include "fhe_precompiles_b200.h"\nint main(void) { fhe_b200_call c; c.op = 0; return (int)sizeof(c) == 0; }\n')
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_rust_shim_lists_every_precompile():
    from fhe_precompiles_b200 import _lib

    text = open(os.path.join(ROOT, "bindings/rust/src/lib.rs")).read()
    for n in _lib.PRECOMPILES:
        assert f"fn c_fhe_{n}(" in text and f"pub fn {n}(&self" in text


def test_header_is_plain_c_and_example_links(tmp_path):
    """include/fhe_precompiles_b200.h must be consumable by a C compiler (the reference's consumers bind it through cgo / C
    shims): examples/c_caller.c builds with -std=c11 -pedantic against the shared library and runs its GPU-free part."""
    import subprocess

    exe = tmp_path / "c_caller"
    lib_dir = os.path.join(ROOT, "fhe_precompiles_b200")
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", "c_caller.c"), "-L" + lib_dir, "-lfhe_precompiles_b200",
                    "-Wl,-rpath," + lib_dir, "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "network public key: 410994 bytes" in r.stdout, r.stdout + r.stderr


def test_sha512_matches_hashlib():
    """the seed of encrypt / reencrypt is SHA-512 of caller data (fhe.rs:600-612): both implementations behind it (built-in and
    libcrypto's when present) against Python's, across the padding boundaries"""
    import ctypes
    import hashlib

    from fhe_precompiles_b200 import _lib

    L = _lib.lib()
    rng = __import__("numpy").random.default_rng(9)
    out = ctypes.create_string_buffer(64)
    for n in [0, 1, 3, 55, 56, 111, 112, 113, 127, 128, 129, 239, 240, 255, 256, 1000, 4097, 500001]:
        data = bytes(rng.integers(0, 256, n, dtype="uint8"))
        for portable in (0, 1):
            L.fhe_b200_sha512(data, n, portable, out)
            assert out.raw == hashlib.sha512(data).digest(), (n, portable)


def test_host_pool_exception_safety(tmp_path):
    """csrc/host_pool.h: a throwing work item reaches the caller of run() (-> code 7 through guarded()), never std::terminate,
    and run() returns only after every copy has finished (tests/host_pool_test.cpp)."""
    import subprocess

    exe = tmp_path / "host_pool_test"
    subprocess.run(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "fhe_precompiles_b200", "csrc"),
                    os.path.join(ROOT, "tests", "host_pool_test.cpp"), "-o", str(exe), "-lpthread"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stdout + r.stderr


def test_data_type_rule_is_exact_per_kind(lib):
    """A ciphertext argument passes iff its data_type equals the string sunscreen 0.8.1 writes for the precompile's type
    (its runtime rejects any other Type -> code 7, fhe.rs:28).  derive(TypeName) drops generic arguments, so Unsigned64 and
    Unsigned256 share one name (pinned by the reference's known answers, tests/test_oracle_kat.py): the first kind that
    carries the name is reported."""
    f = lib.fhe_b200_data_type_kind
    f.argtypes, f.restype = [ctypes.c_char_p], ctypes.c_int32
    from oracle import formats as F

    kinds = {"u256": 0, "u64": 0, "i64": 2, "frac64": 3}
    for k, idx in kinds.items():
        assert f((F.TYPE_NAMES[k] + ",0.8.1,true").encode()) == idx
        assert f((F.TYPE_NAMES[k] + ",0.8.1,false").encode()) == -1  # a plaintext type is not a ciphertext operand
        assert f((F.TYPE_NAMES[k] + ",0.8.0,true").encode()) == -1  # Type equality includes the crate version
    for bad in ("sunscreen::types::bfv::unsigned::Unsigned<2>,0.8.1,true", "sunscreen::types::bfv::unsigned::Unsigned<4>,0.8.1,true",
                "my::Signedish,0.8.1,true", "NotSigned,0.8.1,true", "sunscreen::types::bfv::rational::Rational,0.8.1,true",
                "Signed", "Signed,0.8.1,true", "", "sunscreen::types::bfv::fractional::Fractional<64>,0.8.1,true"):
        assert f(bad.encode()) == -1, bad
