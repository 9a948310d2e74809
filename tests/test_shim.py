"""include/bavoxel_b200.hpp: the reference's C++ call surface (VOX_HESS / BALM2) on top of the C ABI.
CPU: the shim compiles and links in its Eigen-free mode. GPU: the reference call pattern
(benchmark_realworld.cpp:194-218) runs and converges in both precision modes."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "shim_smoke.bin")


def _build():
    lib = os.path.join(ROOT, "balm_b200")
    subprocess.check_call(["g++", "-O1", "-std=c++14", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "shim_smoke.cpp"), "-o", EXE, "-L" + lib, "-lbalm_b200",
                           "-Wl,-rpath," + lib, "-ldl", "-lpthread", "-lrt"])


EXE2 = os.path.join(ROOT, "tests", "shim_eigen_branch.bin")


def _build_eigen_branch():
    lib = os.path.join(ROOT, "balm_b200")
    subprocess.check_call(["g++", "-O1", "-std=c++14", "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(ROOT, "tests", "eigen_stub"),
                           os.path.join(ROOT, "tests", "shim_eigen_branch.cpp"), "-o", EXE2, "-L" + lib, "-lbalm_b200",
                           "-Wl,-rpath," + lib, "-ldl", "-lpthread", "-lrt"])


def test_shim_eigen_branch_compiles_and_links():
    """The BALM_B200_WITH_EIGEN branch (reference types: Eigen::MatrixXd / VectorXd / Matrix3d members) against a stand-in
    for the few Eigen members it uses, and &VOX_HESS::left_evaluate_acc2 handed to std::thread as bavoxel.hpp:1047 does."""
    _build_eigen_branch()
    assert os.path.exists(EXE2)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [0, 1])
def test_reference_divide_thread_left_runs_on_the_shim(prec):
    _build_eigen_branch()
    out = subprocess.run([EXE2, str(prec)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "shim_eigen_branch:" in out.stdout


def test_shim_compiles_and_links():
    _build()
    assert os.path.exists(EXE)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [0, 1])
def test_shim_runs_reference_call_pattern(prec):
    _build()
    out = subprocess.run([EXE, str(prec)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "iter0:" in out.stdout and "shim_smoke: residual" in out.stdout  # the reference's trace line (:1132)


# ---- the shim on top of the REFERENCE'S OWN tools.hpp (PointCluster, IMUST; stand-in Eigen / PCL of oracle/ref_stubs) ----
REF_INC = os.path.join(os.environ.get("BALM_REFERENCE_DIR", "/nonexistent"), "include")
EXE3 = os.path.join(ROOT, "tests", "shim_reference_types.bin")


def build_reference_types():
    lib = os.path.join(ROOT, "balm_b200")
    subprocess.check_call(["g++", "-O1", "-std=c++14", "-w", "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(ROOT, "oracle", "ref_stubs"), "-I" + REF_INC,
                           os.path.join(ROOT, "tests", "shim_reference_types.cpp"), "-o", EXE3, "-L" + lib, "-lbalm_b200",
                           "-Wl,-rpath," + lib, "-ldl", "-lpthread", "-lrt"])


@pytest.mark.skipif(not os.path.exists(os.path.join(REF_INC, "tools.hpp")), reason="BALM_REFERENCE_DIR does not name a checkout of the reference")
def test_shim_compiles_on_the_reference_types():
    """#include "tools.hpp" (the reference's, verbatim) + the shim in BALM_B200_WITH_EIGEN mode with its default plptrs type
    pcl::PointCloud<PointType>::Ptr: what a BALM translation unit looks like after swapping bavoxel.hpp for the shim."""
    build_reference_types()
    assert os.path.exists(EXE3)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [0, 1])
def test_shim_runs_on_the_reference_types(prec):
    if os.path.exists(os.path.join(REF_INC, "tools.hpp")):
        build_reference_types()
    if not os.path.exists(EXE3):
        pytest.skip("tests/shim_reference_types.bin was not built (needs BALM_REFERENCE_DIR at build time)")
    out = subprocess.run([EXE3, str(prec)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "shim_reference_types: residual" in out.stdout
