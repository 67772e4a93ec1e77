"""The grouped extension of the C++ mirror (include/milagro_bls_b200.hpp, AggregateSignature::
verify_multiple_aggregate_signatures_grouped) over b3_verify_multiple_grouped, driven by tests/cpp/test_grouped.cpp.  The non-GPU
test checks that header and program compile and link against the library, and that without a device the program refuses to
run (no CPU path); the GPU test runs it."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_grouped.cpp")
EXE = os.path.join(ROOT, "tests", "cpp", "test_grouped")
HDRS = [os.path.join(ROOT, "include", f) for f in ("milagro_bls_b200.h", "milagro_bls_b200.hpp")]


@pytest.fixture(scope="module")
def exe():
    import __graft_entry__ as g
    lib = g.build_cuda()
    deps = [SRC, lib] + HDRS
    if not os.path.exists(EXE) or any(os.path.getmtime(d) > os.path.getmtime(EXE) for d in deps):
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-o", EXE, SRC, "-L", os.path.dirname(lib), "-lmilagro_bls_b200",
                               "-Wl,-rpath," + os.path.dirname(lib)])
    return EXE


def test_cpp_grouped_compiles_and_refuses_without_a_device(exe):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: see test_cpp_grouped_matches_ungrouped")
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "no CPU path" in out.stdout


@pytest.mark.gpu
def test_cpp_grouped_matches_ungrouped(exe):
    out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "all checks passed" in out.stdout
