"""The range contracts of csrc/modarith.cuh and of the NTT butterflies in csrc/ntt.cuh, checked primitive by primitive.

tests/modarith_probe.cu compiles the headers for sm_100a into one executable linked against the library's context.o and
kernels.o.  On the CPU (--cpu) it checks the host-built twiddle tables, every Shoup pair of DevConsts, the derived
reduction constants and the per-stage bound table.  On the GPU it runs every primitive on crafted and top-of-domain
operands and compares each output with an exact 128-bit reference: congruent, and inside the range its comment states.
The transforms chain those lazy ranges for twelve stages without reducing, so a result one modulus above its range is
harmless where it is made and overflows a word stages later; the end-to-end parity tests cannot place an intermediate
value at the top of a range, this probe does."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "fhe_precompiles_b200", "csrc")
NVCC = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")

MODS = ["q0", "q1", "P", "b0", "b1", "msk"]
SMALL, LARGE, DUAL = MODS[:3], MODS[3:], ["d0", "d1", "d2"]
KN = 4096


def _bfly(mods):
    names = [f"{k}.{m}.G{g}" for m in mods for k in ("fwd_bfly", "inv_bfly") for g in range(12)]
    return names + [f"inv_bfly_last.{m}.{c}" for m in mods for c in ("lazy", "canon")]


def _bfly_prefixes(mods):
    return [f"{k}.{m}." for m in mods for k in ("fwd_bfly", "inv_bfly", "inv_bfly_last")]


SHOUP32 = ([f"shoup32.d_C[{i}]" for i in range(6)] + [f"shoup32.d_W[{i}]" for i in range(4)]
           + [f"shoup32.lk_R[{m}][{i}]" for m in range(3) for i in range(6)]
           + [f"shoup32.tw{t}.s{i}.{k}" for i in range(6) for t in "fi" for k in (1, KN - 1)])

# family -> (--case prefixes, case names the probe must report)
FAMILIES = {
    "shoup": (["shoup_acc", "shoup_lazy", "shoup."],
              [f"shoup_acc0.{m}" for m in MODS] + [f"shoup_acc{k}.{m}" for k in (1, 2) for m in SMALL]
              + [f"shoup_lazy.{m}" for m in MODS] + [f"shoup.{m}" for m in MODS]),
    "dual": (["shoup32.", "barrett61.", "dual_mulsum"],
             SHOUP32 + [f"{k}.s{i}" for k in ("barrett61", "dual_mulsum1", "dual_mulsum2") for i in range(6)]),
    "widesum": (["widesum"], [f"widesum{t}.{m}" for t in (4, 6, 7) for m in SMALL]),
    "mulsum": (["mulsum", "mulmod."],
               [f"mulsum_small{k}.{m}" for k in (1, 2) for m in SMALL] + [f"mulsum_large{k}.{m}" for k in (1, 2) for m in LARGE]
               + [f"mulmod.{m}" for m in MODS]),
    "fold": (["fold", "canon", "reduce64.", "addmod.", "submod.", "mac128"],
             [f"{k}.{m}" for k in ("fold", "fold_k32", "canon", "canon_k32", "reduce64", "addmod", "submod") for m in MODS]
             + ["mac128"]),
    "bfly_small": (_bfly_prefixes(SMALL), _bfly(SMALL)),
    "bfly_large": (_bfly_prefixes(LARGE), _bfly(LARGE)),
    "bfly_dual": (_bfly_prefixes(DUAL), _bfly(DUAL)),
}
LINE = re.compile(r"^case (\S+) evaluated=(\d+) cong_fail=(\d+) range_fail=(\d+) ", re.M)


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    subprocess.run(["make", "-C", CSRC, "build/context.o", "build/kernels.o"], check=True, capture_output=True)
    exe = tmp_path_factory.mktemp("probe") / "modarith_probe"
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-I" + CSRC,
                        os.path.join(ROOT, "tests", "modarith_probe.cu"), os.path.join(CSRC, "build", "context.o"),
                        os.path.join(CSRC, "build", "kernels.o"), "-ldl", "-o", str(exe)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    return str(exe)


def test_host_tables_and_constants(probe):
    r = subprocess.run([probe, "--cpu"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.rstrip().endswith("host ok"), r.stdout + r.stderr
    # every (w, ws) lane of the 18 tables, the pass-9 copies included
    assert "host twiddle_pairs=184320" in r.stdout, r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_primitive_contracts_on_the_gpu(probe, family):
    prefixes, names = FAMILIES[family]
    r = subprocess.run([probe, "--case", ",".join(prefixes)], capture_output=True, text=True, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out
    seen = {m.group(1): tuple(int(x) for x in m.group(2, 3, 4)) for m in LINE.finditer(r.stdout)}
    missing = [n for n in names if n not in seen]
    assert not missing, f"cases not reported: {missing}\n{out}"
    for n in names:
        evaluated, cong, rng = seen[n]
        assert evaluated > 0 and cong == 0 and rng == 0, f"{n}: {seen[n]}\n{out}"
        if n.startswith("shoup32."):
            assert evaluated == 1 << 32, f"{n}: exhaustive sweep evaluated {evaluated}"
