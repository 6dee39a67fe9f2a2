"""Independent numpy restatement of one pcl::CropBox stage (TEST INFRASTRUCTURE ONLY), written apart from the C++
statement in tests/crop_box_oracle.cpp so that the two, and the known answers of tests/golden/crop_box.json, pin each other.
All arithmetic is numpy float32: every `*` and `+` rounds on its own (numpy never contracts to FMA)."""
from __future__ import annotations

import numpy as np

F32 = np.float32


# pcl::CropBox (PCL 1.8.1 filters/impl/crop_box.hpp, CropBox::applyFilter(std::vector<int>&)) ---------------------------
# Semantics (restated from PCL 1.8.1; tests/crop_box_oracle.cpp has the C++ statement of the same function):
#   1. input not dense and x, y or z non-finite -> removed, whatever `negative` is (a filter's output is dense, so with
#      PassThrough stages or an earlier box in front only the segment's own flag can make this step bite);
#   2. local = p; if transform_ is not the identity (Eigen's fuzzy isIdentity, 1e-5): local = transformPoint(local, transform_);
#   3. if translation_ != 0 (exact compare): local -= translation_;
#   4. if rotation_ != 0 (exact compare): inv = getTransformation(0, 0, 0, roll, pitch, yaw).inverse(); if inv is not the
#      identity (fuzzy): local = transformPoint(local, inv);
#   5. outside = any(local < min) or any(local > max); kept iff outside == negative (a NaN coordinate counts as inside).
# transformPoint is ((m00*x + m01*y) + m02*z) + m03 per row, the steps one after another; the cosines and sines are libm's
# float cosf / sinf (numpy's own float32 trig can differ in the last ulp), the inverse is Eigen's 3x3 cofactor formula.
_LIBM = None


def _libm():
    global _LIBM
    if _LIBM is None:
        import ctypes
        import ctypes.util
        lm = ctypes.CDLL(ctypes.util.find_library("m") or "libm.so.6")
        for name in ("cosf", "sinf"):
            getattr(lm, name).restype = ctypes.c_float
            getattr(lm, name).argtypes = [ctypes.c_float]
        _LIBM = lm
    return _LIBM


def is_identity(m) -> bool:
    """Eigen 3.3 MatrixBase::isIdentity(dummy_precision<float>() = 1e-5) of an Affine3f given as its 3x4 rows."""
    m = np.asarray(m, F32).reshape(3, 4)
    prec = F32(1e-5)
    with np.errstate(invalid="ignore"):
        for r in range(3):
            for c in range(4):
                v = m[r, c]
                if r == c:
                    if not (abs(F32(v - F32(1))) <= F32(min(abs(v), F32(1)) * prec)):
                        return False
                elif not (abs(v) <= prec):
                    return False
    return True


def rotation_inverse(roll, pitch, yaw) -> np.ndarray:
    """getTransformation(0, 0, 0, roll, pitch, yaw).inverse() as a 3x4 float32 matrix (Transform::inverse, Affine mode)."""
    lm = _libm()
    cf, sf = (lambda v: F32(lm.cosf(float(F32(v))))), (lambda v: F32(lm.sinf(float(F32(v)))))
    A, B, Cp, D, E, Fr = cf(yaw), sf(yaw), cf(pitch), sf(pitch), cf(roll), sf(roll)
    with np.errstate(all="ignore"):
        DE, DF = F32(D * E), F32(D * Fr)
        R = np.array([[A * Cp, F32(A * DF) - F32(B * E), F32(B * Fr) + F32(A * DE)],
                      [B * Cp, F32(A * E) + F32(B * DF), F32(B * DE) - F32(A * Fr)],
                      [-D, Cp * Fr, Cp * E]], F32)

        def cof(i, j):
            i1, i2, j1, j2 = (i + 1) % 3, (i + 2) % 3, (j + 1) % 3, (j + 2) % 3
            return F32(F32(R[i1, j1] * R[i2, j2]) - F32(R[i1, j2] * R[i2, j1]))
        det = F32(F32(F32(cof(0, 0) * R[0, 0]) + F32(cof(1, 0) * R[1, 0])) + F32(cof(2, 0) * R[2, 0]))
        invdet = F32(F32(1) / det)
        out = np.zeros((3, 4), F32)
        for i in range(3):
            for j in range(3):
                out[i, j] = F32(cof(j, i) * invdet)
            # translation column: (-linear) * (0, 0, 0): a signed zero (NaN for a non-finite linear part)
            z = F32(0)
            out[i, 3] = F32(F32(F32(-out[i, 0]) * z) + F32(F32(-out[i, 1]) * z)) + F32(F32(-out[i, 2]) * z)
    return out


def crop_box_mask(xyzi: np.ndarray, is_dense: bool, box: dict) -> np.ndarray:
    """One CropBox stage -> boolean keep mask. box: dict(min, max, translation, rotation, transform (3x4), negative)."""
    p = np.asarray(xyzi, F32).reshape(-1, 4)
    x, y, z = p[:, 0].copy(), p[:, 1].copy(), p[:, 2].copy()
    keep = np.ones(len(p), bool)
    if not is_dense:
        keep &= np.isfinite(x) & np.isfinite(y) & np.isfinite(z)
    with np.errstate(all="ignore"):
        def apply(m, x, y, z):
            return tuple(((m[r, 0] * x + m[r, 1] * y) + m[r, 2] * z) + m[r, 3] for r in range(3))
        t = np.asarray(box.get("transform", np.eye(3, 4)), F32).reshape(3, 4)
        if not is_identity(t):
            x, y, z = apply(t, x, y, z)
        tr = np.asarray(box.get("translation", (0, 0, 0)), F32)
        if (tr != 0).any():
            x, y, z = x - tr[0], y - tr[1], z - tr[2]
        rot = np.asarray(box.get("rotation", (0, 0, 0)), F32)
        if (rot != 0).any():
            inv = rotation_inverse(*rot)
            if not is_identity(inv):
                x, y, z = apply(inv, x, y, z)
        mn, mx = np.asarray(box["min"], F32), np.asarray(box["max"], F32)
        outside = (x < mn[0]) | (y < mn[1]) | (z < mn[2]) | (x > mx[0]) | (y > mx[1]) | (z > mx[2])
    return keep & (outside == bool(box.get("negative", False)))


def crop_boxes(xyzi: np.ndarray, keep: np.ndarray, is_dense: bool, passes_in_front: bool, boxes) -> np.ndarray:
    """The CropBox stages after a PassThrough chain: `keep` is the chain's mask; each box filters the previous output."""
    keep = keep.copy()
    dense = bool(is_dense) or passes_in_front
    for b in boxes:
        sel = np.nonzero(keep)[0]
        keep[sel] = crop_box_mask(xyzi[sel], dense, b)
        dense = True
    return keep
