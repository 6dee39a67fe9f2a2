"""ctypes binding of tests/plane_axis_oracle.cpp, the C++ statement of pcl::SACSegmentation with SACMODEL_PLANE,
SACMODEL_PERPENDICULAR_PLANE and SACMODEL_PARALLEL_PLANE (TEST INFRASTRUCTURE ONLY), and of tests/plane_axis_pcl_ref.cpp,
the real PCL behind the same signature where PCL is installed. Compiled on first use into a per-user temporary directory,
so the repository tree is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess

import numpy as np

from crop_box_oracle import _build

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        # the source includes oracle/cm_oracle.cpp: its hash keys the build too
        base = open(os.path.join(os.path.dirname(HERE), "oracle", "cm_oracle.cpp"), "rb").read()
        _LIB = C.CDLL(_build(os.path.join(HERE, "plane_axis_oracle.cpp"),
                             ["-DCM_ORACLE_SOURCE_%s" % hashlib.sha256(base).hexdigest()[:16]]))
        _LIB.cmo_plane_ransac_model.restype = C.c_int64
    return _LIB


def plane_ransac_model(xyzi: np.ndarray, threshold: float, probability: float = 0.99, max_iterations: int = 1000,
                       optimize: bool = True, seed: int = 12345, sum_order: int = 0, model: int = 0, axis=(0.0, 0.0, 1.0),
                       eps_angle: float = 0.0) -> dict:
    """segment() with setModelType(model) (0 PLANE, 1 PERPENDICULAR_PLANE, 2 PARALLEL_PLANE), setAxis(axis),
    setEpsAngle(eps_angle): the dict of oracle/cm_oracle_py.plane_ransac plus "rejected", the iterations whose model
    failed the axis test."""
    xyzi = np.ascontiguousarray(xyzi, np.float32).reshape(-1, 4)
    n = len(xyzi)
    info = np.zeros(8, np.int32)
    c_r = np.zeros(4, np.float32)
    c_o = np.zeros(4, np.float32)
    inl = np.empty(max(n, 1), np.int32)
    ax = np.ascontiguousarray(np.asarray(axis, np.float32).reshape(3))
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    k = lib().cmo_plane_ransac_model(p(xyzi), C.c_int64(n), C.c_double(threshold), C.c_double(probability), int(max_iterations),
                                     int(bool(optimize)), C.c_uint32(seed), int(sum_order), int(model), p(ax),
                                     C.c_double(eps_angle), p(info), p(c_r), p(c_o), p(inl))
    return {"found": bool(info[0]), "iterations": int(info[1]), "draws": int(info[2]), "best_count": int(info[3]),
            "sample": info[4:7].copy(), "rejected": int(info[7]), "coeff_ransac": c_r, "coeff": c_o,
            "inliers": inl[:k].copy()}


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
        m = ["pcl_segmentation-" + ver, "pcl_sample_consensus-" + ver, "pcl_common-" + ver, "eigen3"]
        if subprocess.run(["pkg-config", "--exists"] + m).returncode == 0:
            mods = m
            break
    if mods is None:
        _WHY = "PCL >= 1.8 not found by pkg-config (pcl_segmentation)"
        return False
    flags = subprocess.run(["pkg-config", "--cflags", "--libs"] + mods, capture_output=True, text=True).stdout.split()
    try:
        L = C.CDLL(_build(os.path.join(HERE, "plane_axis_pcl_ref.cpp"), flags))
    except Exception as e:  # noqa: BLE001 -- reported as the skip reason
        _WHY = "building tests/plane_axis_pcl_ref.cpp failed: %s" % (getattr(e, "stderr", "") or e)[-400:]
        return False
    L.cmp_plane_ransac_model.restype = C.c_int64
    _PCL = L
    return True


def pcl_why_not() -> str:
    return _WHY or "the real-PCL SACSegmentation wrapper is not built"


def pcl_plane_ransac_model(xyzi, threshold, probability=0.99, max_iterations=1000, optimize=True, model=0, axis=(0.0, 0.0, 1.0),
                           eps_angle=0.0):
    """pcl::SACSegmentation itself: (coefficients [4] float32, inlier indices)."""
    xyzi = np.ascontiguousarray(xyzi, np.float32).reshape(-1, 4)
    coeff = np.zeros(4, np.float32)
    inl = np.empty(max(len(xyzi), 1), np.int32)
    ax = np.ascontiguousarray(np.asarray(axis, np.float32).reshape(3))
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    k = _PCL.cmp_plane_ransac_model(p(xyzi), C.c_int64(len(xyzi)), C.c_double(threshold), C.c_double(probability),
                                    int(max_iterations), int(bool(optimize)), int(model), p(ax), C.c_double(eps_angle),
                                    p(coeff), p(inl))
    return coeff, inl[:k].copy()
