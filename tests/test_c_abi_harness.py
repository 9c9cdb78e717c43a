"""Builds tests/c_abi_harness.c with gcc against include/pa_b200.h and
libpa_b200.so and runs it: the boundary used from plain C, without Python or
torch.  On a GPU box it must verify x->y->z bit-exactly (exit 0); on a CPU box
the library must refuse the data path (exit 2: PA_ENOGPU, no CPU fallback)."""
import os
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "pencilarrays.jl_b200")


def _build(tmp_path):
    exe = str(tmp_path / "c_abi_harness")
    cmd = ["/usr/bin/gcc", "-std=c11", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
           "-I", "/usr/local/cuda/include", os.path.join(ROOT, "tests", "c_abi_harness.c"), "-o", exe,
           "-L", PKG, "-l:libpa_b200.so", "-L", "/usr/local/cuda/lib64", "-lcudart",
           f"-Wl,-rpath,{PKG}", "-Wl,-rpath,/usr/local/cuda/lib64"]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return exe


def test_c_harness_refuses_without_gpu(tmp_path):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    out = subprocess.run([_build(tmp_path), str(tmp_path / "io.bin")], capture_output=True, text=True,
                         timeout=120)
    assert out.returncode == 2, (out.stdout, out.stderr)
    assert "no CUDA device" in out.stdout


@pytest.mark.gpu
def test_c_harness_on_gpu(tmp_path):
    out = subprocess.run([_build(tmp_path), str(tmp_path / "io.bin")], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode == 0, (out.stdout, out.stderr)
    assert "C ABI harness OK" in out.stdout
