"""ctypes binding of tests/sor_oracle.cpp, the C++ statement of pcl::StatisticalOutlierRemoval (TEST INFRASTRUCTURE ONLY).
Compiled on first use, with the flags of oracle/Makefile, into a per-user directory under the system temporary directory,
so the repository tree is never written."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

from crop_box_oracle import _build

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class CmoSorStats(C.Structure):
    _fields_ = [("mean", C.c_double), ("stddev", C.c_double), ("threshold", C.c_double), ("sum", C.c_double),
                ("sq_sum", C.c_double), ("n_valid", C.c_int64), ("too_few", C.c_int32), ("n_kept", C.c_int32)]


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(_build(os.path.join(HERE, "sor_oracle.cpp")))
        _LIB.cmo_statistical_outlier.restype = C.c_int
        _LIB.cmo_statistical_outlier.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_int, C.c_int,
                                                 C.c_void_p, C.c_void_p, C.POINTER(CmoSorStats)]
    return _LIB


def statistical_outlier(xyzi, mean_k: int, std_mul: float, negative: bool = False, sqrt_mode: int = 0) -> dict:
    """the same dict as sor_np.sor_cloud"""
    a = np.ascontiguousarray(np.asarray(xyzi, np.float32).reshape(-1, 4))
    n = len(a)
    dist = np.zeros(max(n, 1), np.float32)
    keep = np.zeros(max(n, 1), np.uint8)
    st = CmoSorStats()
    rc = lib().cmo_statistical_outlier(a.ctypes.data_as(C.c_void_p), n, int(mean_k), float(std_mul), int(bool(negative)),
                                       int(sqrt_mode), dist.ctypes.data_as(C.c_void_p), keep.ctypes.data_as(C.c_void_p),
                                       C.byref(st))
    assert rc == 0
    return {"distances": dist[:n], "keep": keep[:n].astype(bool), "mean": st.mean, "stddev": st.stddev,
            "threshold": st.threshold, "n_valid": int(st.n_valid), "too_few": bool(st.too_few), "sum": st.sum,
            "sq_sum": st.sq_sum}


# ---- the real PCL ------------------------------------------------------------------------------------------------------------
_PCL = None
_WHY = ""


def pcl_available() -> bool:
    """Builds the real-PCL wrapper when pkg-config finds PCL's filters module (>= 1.8); never raises."""
    global _PCL, _WHY
    if _PCL is not None:
        return True
    if not shutil.which("pkg-config"):
        _WHY = "pkg-config not found"
        return False
    mods = None
    for ver in ("1.8", "1.9", "1.10", "1.11", "1.12", "1.13", "1.14"):
        m = ["pcl_filters-" + ver, "pcl_search-" + ver, "pcl_kdtree-" + ver, "pcl_common-" + ver, "eigen3"]
        if subprocess.run(["pkg-config", "--exists"] + m).returncode == 0:
            mods = m
            break
    if mods is None:
        _WHY = "PCL >= 1.8 not found by pkg-config (pcl_filters)"
        return False
    flags = subprocess.run(["pkg-config", "--cflags", "--libs"] + mods, capture_output=True, text=True).stdout.split()
    try:
        L = C.CDLL(_build(os.path.join(HERE, "sor_pcl_ref.cpp"), flags))
    except Exception as e:  # noqa: BLE001 -- reported as the skip reason
        _WHY = "building tests/sor_pcl_ref.cpp failed: %s" % (getattr(e, "stderr", "") or e)[-400:]
        return False
    L.cmp_statistical_outlier.restype = C.c_int64
    L.cmp_statistical_outlier.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_int32, C.c_void_p]
    _PCL = L
    return True


def pcl_why_not() -> str:
    return _WHY or "the real-PCL StatisticalOutlierRemoval wrapper is not built"


def pcl_statistical_outlier(xyzi, mean_k: int, std_mul: float, negative: bool = False) -> np.ndarray:
    """pcl::StatisticalOutlierRemoval itself: indices kept, in input order."""
    a = np.ascontiguousarray(np.asarray(xyzi, np.float32).reshape(-1, 4))
    out = np.zeros(max(len(a), 1), np.int32)
    k = _PCL.cmp_statistical_outlier(a.ctypes.data_as(C.c_void_p), len(a), int(mean_k), float(std_mul), int(bool(negative)),
                                     out.ctypes.data_as(C.c_void_p))
    return out[:k].astype(np.int64)
