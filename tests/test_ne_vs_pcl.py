"""The C++ statement of pcl::NormalEstimation (tests/ne_oracle.cpp) against the REAL class (tests/ne_pcl_ref.cpp) with a
tolerance: the statement uses the library's trig rule, PCL the host libm (DESIGN section 8), so the bits may differ.
Where PCL is not installed (this repository's build image) these tests SKIP and say why; where pkg-config finds
PCL >= 1.8 the wrapper is built on first use."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import ne_cases as K
import ne_oracle as O
from crop_box_oracle import _build

HERE = os.path.dirname(os.path.abspath(__file__))


def _pcl():
    if not shutil.which("pkg-config"):
        return None, "pkg-config not found"
    for ver in ("1.8", "1.9", "1.10", "1.11", "1.12", "1.13", "1.14"):
        m = ["pcl_features-" + ver, "pcl_search-" + ver, "pcl_kdtree-" + ver, "pcl_common-" + ver, "eigen3"]
        if subprocess.run(["pkg-config", "--exists"] + m).returncode == 0:
            flags = subprocess.run(["pkg-config", "--cflags", "--libs"] + m, capture_output=True, text=True).stdout.split()
            try:
                L = C.CDLL(_build(os.path.join(HERE, "ne_pcl_ref.cpp"), flags))
            except Exception as e:  # noqa: BLE001 -- reported as the skip reason
                return None, "building tests/ne_pcl_ref.cpp failed: %s" % (getattr(e, "stderr", "") or e)[-400:]
            L.cmp_normals.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_void_p]
            return L, ""
    return None, "PCL >= 1.8 not found by pkg-config (pcl_features)"


PCL, WHY = _pcl()
pytestmark = pytest.mark.skipif(PCL is None, reason="real-PCL NormalEstimation not available: " + WHY)


@pytest.mark.parametrize("radius", [0.1, 0.3, 0.5])
def test_normals_match_pcl(radius):
    for x in (K.roi_cloud(7, 32, 1024), K.eigen_family(1, 0.3), K.small_groups(0.3), K.lattice(8, 0.25)):
        a = np.ascontiguousarray(x, np.float32)
        vp = np.array([0.0, 0.0, 1.8], np.float32)
        got = np.zeros((len(a), 4), np.float32)
        PCL.cmp_normals(a.ctypes.data_as(C.c_void_p), len(a), radius, vp.ctypes.data_as(C.c_void_p),
                        got.ctypes.data_as(C.c_void_p))
        want = O.normals(a, radius, vp)
        assert (np.isnan(got[:, 0]) == np.isnan(want[:, 0])).all()
        ok = ~np.isnan(want[:, 0])
        assert np.abs(got[ok] - want[ok]).max() < 1e-2
        assert (np.abs(got[ok] - want[ok]).max(axis=1) < 1e-5).mean() > 0.95
