"""numpy restatement of the axis test of SACMODEL_PERPENDICULAR_PLANE / SACMODEL_PARALLEL_PLANE (PCL 1.8.1 isModelValid)
and of RandomSampleConsensus::computeModel with it (TEST INFRASTRUCTURE ONLY), written independently of
tests/plane_axis_oracle.cpp so that the two pin each other. Sampler, model and score are oracle/np_oracle.py's. The double
angle uses math.acos / math.sin (the libm, as PCL does): numpy's vectorised arccos may differ in the last bit."""
from __future__ import annotations

import math

import numpy as np

from oracle import np_oracle as NP

F32 = np.float32
INT32_MAX = 2**31 - 1


def normalize4(v, order: int):
    """Eigen 3.3 normalize() of a Vector4f: divides only when the squared norm is positive."""
    v = np.asarray(v, F32).copy()
    with np.errstate(all="ignore"):
        z = NP._sum4(v[0] * v[0], v[1] * v[1], v[2] * v[2], v[3] * v[3], order)
        if z > 0:
            v = (v / np.sqrt(z, dtype=F32)).astype(F32)
    return v


def plane_axis_dot(c, model: int, axis, order: int = 0):
    """The float d of isModelValid: (a, b, c, 0) normalized (twice for PERPENDICULAR, the second time in getAngle3D)
    dotted with (ax, ay, az, 0) normalized."""
    m = normalize4([c[0], c[1], c[2], 0.0], order)
    if model == 1:
        m = normalize4(m, order)
    a = normalize4([axis[0], axis[1], axis[2], 0.0], order)
    with np.errstate(all="ignore"):
        return F32(NP._sum4(a[0] * m[0], a[1] * m[1], a[2] * m[2], a[3] * m[3], order))


def perpendicular_angle(d) -> float:
    """min(angle, pi - angle) of SACMODEL_PERPENDICULAR_PLANE for the float d (getAngle3D: clamp to [-1, 1], acos)."""
    rad = float(d)
    if rad != rad:
        return float("nan")
    rad = -1.0 if rad < -1.0 else 1.0 if rad > 1.0 else rad
    angle = abs(math.acos(rad))
    return min(angle, math.pi - angle)


def plane_model_valid(c, model: int = 0, axis=(0.0, 0.0, 1.0), eps_angle: float = 0.0, order: int = 0) -> bool:
    """isModelValid of SACMODEL_PLANE (0), PERPENDICULAR_PLANE (1) and PARALLEL_PLANE (2): tested only when
    eps_angle > 0; a NaN model passes (every comparison with NaN is false)."""
    if model == 0 or not eps_angle > 0.0:
        return True
    d = plane_axis_dot(c, model, axis, order)
    if model == 1:
        return not perpendicular_angle(d) > eps_angle
    return not float(abs(d)) > abs(math.sin(eps_angle))


def plane_ransac(xyzi: np.ndarray, threshold: float, probability: float = 0.99, max_iterations: int = 1000,
                 seed: int = 12345, order: int = 0, model: int = 0, axis=(0.0, 0.0, 1.0), eps_angle: float = 0.0) -> dict:
    """computeModel with the axis test, no refit. A model that fails it counts 0 inliers and is still an iteration
    ("rejected" counts them); "best_valid": whether the returned model passes it (if not, selectWithinDistance keeps
    no point)."""
    x = np.ascontiguousarray(xyzi, F32).reshape(-1, 4)
    n = len(x)
    out = {"found": False, "iterations": 0, "draws": 0, "best_count": 0, "sample": np.full(3, -1, np.int32),
           "coeff": np.zeros(4, F32), "rejected": 0, "best_valid": False}
    if n < 3:
        return out
    raw = np.random.RandomState(seed)._bit_generator
    shuffled = np.arange(n, dtype=np.int64)
    iterations, draws, best, k = 0, 0, -INT32_MAX, 1.0
    with np.errstate(divide="ignore", invalid="ignore"):
        log_p = np.log(1.0 - probability)
    while iterations < k:
        got = False
        for _ in range(1000):
            for i in range(3):
                r = int(raw.random_raw()) >> 1
                j = i + r % (n - i)
                shuffled[i], shuffled[j] = shuffled[j], shuffled[i]
            draws += 1
            sel = shuffled[:3].copy()
            good, c = NP.plane_of_sample(x[sel[0]], x[sel[1]], x[sel[2]], order)
            if good:
                got = True
                break
        if not got:
            break
        valid = plane_model_valid(c, model, axis, eps_angle, order)
        out["rejected"] += 0 if valid else 1
        cnt = int(NP.plane_inlier_mask(x, c, threshold, order).sum()) if valid else 0
        if cnt > best:
            best = cnt
            out.update(found=True, best_count=cnt, sample=sel.astype(np.int32), coeff=c.copy(), best_valid=valid)
            w = best / n
            p_no = 1.0 - w ** 3.0
            p_no = min(max(np.finfo(np.float64).eps, p_no), 1.0 - np.finfo(np.float64).eps)
            k = log_p / np.log(p_no)
        iterations += 1
        if iterations > max_iterations:
            break
    out.update(iterations=iterations, draws=draws)
    return out
