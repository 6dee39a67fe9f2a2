"""ctypes binding of tests/ne_oracle.cpp, the C++ statement of pcl::NormalEstimation with a radius search, and of the
checks of the trig rule (TEST INFRASTRUCTURE ONLY). Compiled on first use, with the flags of oracle/Makefile plus -pthread,
into a per-user directory under the system temporary directory (keyed by the source, cm_ne_math.h and the flags), so the
repository tree is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os

import numpy as np

from crop_box_oracle import _build

HERE = os.path.dirname(os.path.abspath(__file__))
MATH_H = os.path.join(os.path.dirname(HERE), "cloud_merger_b200", "csrc", "cm_ne_math.h")
F32 = np.float32
QNAN_BITS = 0x7FC00000
# cm_ne_math.h's PATH_* bits
ROOTS2, TRIG, Q_CLAMP, ROOT0_NEG, PICK1, PICK2, PICK3, NAN_COV, FLIP = 1, 2, 4, 8, 16, 32, 64, 128, 256
_LIB = None
_P = C.c_void_p


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        tag = hashlib.sha256(open(MATH_H, "rb").read()).hexdigest()[:16]  # _build keys on the source text only
        L = C.CDLL(_build(os.path.join(HERE, "ne_oracle.cpp"), ["-pthread", "-DCM_NE_MATH_TAG=" + tag]))
        L.cmo_normals.argtypes = [_P, C.c_int64, C.c_double, _P, C.c_int, C.c_int, _P, _P, _P, _P]
        L.cmo_solve.argtypes = [_P, _P, _P, C.c_int64, _P, C.c_int, _P, _P]
        for f in ("cmo_cos", "cmo_sin"):
            getattr(L, f).argtypes = [C.c_float]
            getattr(L, f).restype = C.c_float
        L.cmo_atan2.argtypes = [C.c_float, C.c_float]
        L.cmo_atan2.restype = C.c_float
        L.cmo_sincos_check.argtypes = [C.c_uint32, C.c_uint32, _P]
        L.cmo_atan2_check.argtypes = [C.c_uint64, C.c_int64, _P]
        L.cmo_set_threads.argtypes = [C.c_int]
        L.cmo_set_threads.restype = None
        _LIB = L
    return _LIB


def _ptr(a):
    return a.ctypes.data_as(_P)


def _vp(viewpoint):
    return np.asarray(viewpoint, F32).reshape(3)


def normals(xyzi, radius: float, viewpoint=(0.0, 0.0, 0.0), trig_mode: int = 0, exhaustive: bool = False,
            details: bool = False):
    """PCL's normals of one cloud: float32 [n, 4] (nx ny nz curvature, input order). details: also the neighbourhood
    sizes, the PATH_* bits and the scaled covariance's roots of every point."""
    a = np.ascontiguousarray(np.asarray(xyzi, F32).reshape(-1, 4))
    n = len(a)
    out = np.zeros((max(n, 1), 4), F32)
    cnt = np.zeros(max(n, 1), np.int32)
    paths = np.zeros(max(n, 1), np.uint32)
    roots = np.zeros((max(n, 1), 3), F32)
    vp = _vp(viewpoint)
    assert lib().cmo_normals(_ptr(a), n, float(radius), _ptr(vp), int(trig_mode), int(bool(exhaustive)), _ptr(out),
                             _ptr(cnt), _ptr(paths), _ptr(roots)) == 0
    if details:
        return out[:n], cnt[:n], paths[:n], roots[:n]
    return out[:n]


def set_threads(n: int) -> None:
    """threads of the statement's point loop: 1 for a one-core timing, 0 for one per hardware thread"""
    lib().cmo_set_threads(int(n))


def solve(sums, counts, xyzi, viewpoint=(0.0, 0.0, 0.0), trig_mode: int = 0):
    """cm_ne_math.h's solve on given running sums [n, 9] (float32), counts and query points: ([n, 4], PATH_* bits)."""
    s = np.ascontiguousarray(np.asarray(sums, F32).reshape(-1, 9))
    c = np.ascontiguousarray(np.asarray(counts, np.int64))
    q = np.ascontiguousarray(np.asarray(xyzi, F32).reshape(-1, 4))
    n = len(s)
    out = np.zeros((max(n, 1), 4), F32)
    paths = np.zeros(max(n, 1), np.uint32)
    vp = _vp(viewpoint)
    assert lib().cmo_solve(_ptr(s), _ptr(c), _ptr(q), n, _ptr(vp), int(trig_mode), _ptr(out), _ptr(paths)) == 0
    return out[:n], paths[:n]


def atan2(y, x):
    return F32(lib().cmo_atan2(float(y), float(x)))


def cos(x):
    return F32(lib().cmo_cos(float(x)))


def sin(x):
    return F32(lib().cmo_sin(float(x)))


def sincos_check(lo_bits: int, hi_bits: int) -> dict:
    st = np.zeros(7, np.int64)
    assert lib().cmo_sincos_check(lo_bits, hi_bits, _ptr(st)) == 0
    return dict(zip(("floats", "sin_bad", "cos_bad", "unresolved", "sinf_same", "cosf_same", "sign_bad"), st.tolist()))


def atan2_check(seed: int, n: int) -> dict:
    st = np.zeros(4, np.int64)
    assert lib().cmo_atan2_check(seed, n, _ptr(st)) == 0
    return dict(zip(("samples", "bad", "unresolved", "atan2f_same"), st.tolist()))
