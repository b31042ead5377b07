"""integration/src/ace_b200_shim.cpp -- the Rcpp file a maintainer drops into the R package -- is real code: it is
compiled here against the stand-in RcppArmadillo headers (oracle/miniarma; R / Rcpp / Armadillo are not installed),
linked with libace_b200.so and called the way R calls the exported functions (tests/c/shim_harness.cpp)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "integration", "src", "ace_b200_shim.cpp")


def _build(tmp_path):
    from additivecausalexpansion_b200 import _lib

    _lib.lib()
    libdir = os.path.dirname(_lib.SO_PATH)
    exe = str(tmp_path / "shim_harness")
    cmd = ["g++", "-O1", "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "oracle", "miniarma"), "-I",
           os.path.join(ROOT, "include"), SHIM, os.path.join(ROOT, "tests", "c", "shim_harness.cpp"), "-o", exe,
           "-L", libdir, "-l:libace_b200.so", f"-Wl,-rpath,{libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_shim_exports_the_19_reference_routines():
    """Same names as the reference registers (src/RcppExports.cpp:301-327)."""
    src = open(SHIM).read()
    exported = set(re.findall(r"// \[\[Rcpp::export\]\]\n(?:[\w:<>&\s\*]+?)\s(\w+)\(", src))
    reference = {"kernmat_Matern32_cpp", "kernmat_Matern32_symmetric_cpp", "grad_Matern_cpp", "kernmat_SE_cpp",
                 "kernmat_SE_symmetric_cpp", "invkernel_cpp", "grad_SE_cpp", "ncs_basis", "ncs_basis_deriv",
                 "Nesterov_cpp", "Nadam_cpp", "Adam_cpp", "pred_cpp", "pred_marginal_cpp", "stats_cpp",
                 "mu_solution_cpp", "normalize_train", "normalize_test", "norm_clip_cpp"}
    assert reference <= exported, reference - exported


def test_shim_compiles_and_host_routines_work(tmp_path):
    exe = _build(tmp_path)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.startswith("OK host"), out.stdout + out.stderr


@pytest.mark.gpu
def test_shim_drives_the_gpu_path(tmp_path):
    exe = _build(tmp_path)
    out = subprocess.run([exe, "gpu"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "OK gpu" in out.stdout, out.stdout + out.stderr
