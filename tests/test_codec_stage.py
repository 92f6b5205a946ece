"""csrc/codec_stage.h: the job layout the byte surface's tiles and single calls and upload_ciphertexts share, checked on the CPU
(tests/codec_stage_test.cpp, built with g++ alone)."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INCLUDE = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")  # codec_kernels.h includes cuda_runtime.h


def test_codec_stage_layout(tmp_path):
    exe = tmp_path / "codec_stage_test"
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "fhe_precompiles_b200", "csrc"),
                    "-I" + CUDA_INCLUDE, os.path.join(ROOT, "tests", "codec_stage_test.cpp"), "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stdout + r.stderr
