"""ctypes binding of tests/ec_oracle.cpp, the C++ statement of pcl::EuclideanClusterExtraction (TEST INFRASTRUCTURE ONLY).
Compiled on first use, with the flags of oracle/Makefile, into a per-user directory under the system temporary directory,
so the repository tree is never written. Also builds the real-PCL wrapper tests/ec_pcl_ref.cpp where PCL is installed."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

from crop_box_oracle import _build

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
INT_MAX = 2 ** 31 - 1


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(_build(os.path.join(HERE, "ec_oracle.cpp")))
        _LIB.cmo_euclidean_clusters.restype = C.c_int
        _LIB.cmo_euclidean_clusters.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_int32, C.c_int32, C.c_void_p,
                                                C.c_void_p, C.POINTER(C.c_int64)]
        _LIB.cmo_pcl_cluster_order.restype = C.c_int
        _LIB.cmo_pcl_cluster_order.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
    return _LIB


def euclidean_clusters(xyzi, tolerance: float, min_size: int = 1, max_size: int = INT_MAX) -> list:
    """PCL's clusters of one cloud, in PCL's order: a list of int64 index arrays (ascending inside a cluster)."""
    a = np.ascontiguousarray(np.asarray(xyzi, np.float32).reshape(-1, 4))
    n = len(a)
    idx = np.zeros(max(n, 1), np.int64)
    begin = np.zeros(n + 1, np.int64)
    k = C.c_int64()
    rc = lib().cmo_euclidean_clusters(a.ctypes.data_as(C.c_void_p), n, float(tolerance), int(min_size), int(max_size),
                                      idx.ctypes.data_as(C.c_void_p), begin.ctypes.data_as(C.c_void_p), C.byref(k))
    assert rc == 0
    return [idx[begin[j]:begin[j + 1]].copy() for j in range(k.value)]


def pcl_cluster_order(sizes) -> np.ndarray:
    """std::sort(v.rbegin(), v.rend(), size <) of libstdc++ on clusters of these sizes: input position per rank."""
    s = np.ascontiguousarray(np.asarray(sizes, np.int64))
    out = np.zeros(max(len(s), 1), np.int64)
    assert lib().cmo_pcl_cluster_order(s.ctypes.data_as(C.c_void_p), len(s), out.ctypes.data_as(C.c_void_p)) == 0
    return out[:len(s)]


# ---- the real PCL ------------------------------------------------------------------------------------------------------------
_PCL = None
_WHY = ""


def pcl_available() -> bool:
    """Builds the real-PCL wrapper when pkg-config finds PCL's segmentation module (>= 1.8); never raises."""
    global _PCL, _WHY
    if _PCL is not None:
        return True
    if not shutil.which("pkg-config"):
        _WHY = "pkg-config not found"
        return False
    mods = None
    for ver in ("1.8", "1.9", "1.10", "1.11", "1.12", "1.13", "1.14"):
        m = ["pcl_segmentation-" + ver, "pcl_search-" + ver, "pcl_kdtree-" + ver, "pcl_common-" + ver, "eigen3"]
        if subprocess.run(["pkg-config", "--exists"] + m).returncode == 0:
            mods = m
            break
    if mods is None:
        _WHY = "PCL >= 1.8 not found by pkg-config (pcl_segmentation)"
        return False
    flags = subprocess.run(["pkg-config", "--cflags", "--libs"] + mods, capture_output=True, text=True).stdout.split()
    try:
        L = C.CDLL(_build(os.path.join(HERE, "ec_pcl_ref.cpp"), flags))
    except Exception as e:  # noqa: BLE001 -- reported as the skip reason
        _WHY = "building tests/ec_pcl_ref.cpp failed: %s" % (getattr(e, "stderr", "") or e)[-400:]
        return False
    L.cmp_euclidean_clusters.restype = C.c_int64
    L.cmp_euclidean_clusters.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    _PCL = L
    return True


def pcl_why_not() -> str:
    return _WHY or "the real-PCL EuclideanClusterExtraction wrapper is not built"


def pcl_euclidean_clusters(xyzi, tolerance: float, min_size: int = 1, max_size: int = INT_MAX) -> list:
    """pcl::EuclideanClusterExtraction itself: the clusters as int64 index arrays, in its order."""
    a = np.ascontiguousarray(np.asarray(xyzi, np.float32).reshape(-1, 4))
    idx = np.zeros(max(len(a), 1), np.int64)
    begin = np.zeros(len(a) + 1, np.int64)
    k = _PCL.cmp_euclidean_clusters(a.ctypes.data_as(C.c_void_p), len(a), float(tolerance), int(min_size), int(max_size),
                                    idx.ctypes.data_as(C.c_void_p), begin.ctypes.data_as(C.c_void_p))
    return [idx[begin[j]:begin[j + 1]].copy() for j in range(k)]
