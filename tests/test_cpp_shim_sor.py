"""The statistical outlier removal of the reference-facing C++ shim: builds tests/cpp/test_shim_sor.cpp (with the shim's
ROS / Eigen / tf stand-ins and the C++ statement tests/sor_oracle.cpp) into a temporary directory and runs it.
CPU box: the binary must refuse to compute (exit 77). GPU box: statisticalOutlierRemoval and
Context::statistical_outlier_multi match the statement bit for bit."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP = os.path.join(ROOT, "tests", "cpp")
LIBDIR = os.path.join(ROOT, "cloud_merger_b200")


def _build(tmp_path):
    from cloud_merger_b200 import build as cm_build
    cm_build.build()
    exe = str(tmp_path / "test_shim_sor")
    cmd = [os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra",
           "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(CPP, "mock"),
           os.path.join(CPP, "test_shim_sor.cpp"), os.path.join(ROOT, "tests", "sor_oracle.cpp"), "-o", exe,
           "-L" + LIBDIR, "-lcloud_merger_gpu", "-Wl,-rpath," + LIBDIR, "-lpthread", "-ldl", "-lrt"]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return exe


def test_shim_sor_builds_and_refuses_without_gpu(tmp_path):
    exe = _build(tmp_path)
    from cloud_merger_b200 import _lib
    if _lib.load().cm_device_count() > 0:
        pytest.skip("a GPU is present")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 77, r.stdout + r.stderr
    assert "no CPU path" in r.stdout


@pytest.mark.gpu
def test_shim_sor_matches_statement_on_gpu(gpu_ok, tmp_path):
    exe = _build(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "shim sor ok" in r.stdout
