"""Independent numpy restatement of the merge hot path (TEST INFRASTRUCTURE ONLY).

PARITY UNPINNED: the reference has no tests or golden vectors and its arithmetic lives in PCL 1.8.1 / pcl_ros / Eigen,
which are neither under /root/reference nor installed here (SURVEY.md section 8c). This file restates the published
PCL 1.8.1 algorithms a second time, vectorised and written independently of oracle/cm_oracle.cpp, so that the two
restatements pin each other and the hand-checkable known-answer vector (tests/golden/known_answer.json).

All arithmetic is numpy float32: every `*` and `+` below rounds on its own (numpy never contracts to FMA).
Only tests/ may import this module.
"""
from __future__ import annotations

import numpy as np

F32 = np.float32
INT32_MAX = 2**31 - 1


def unpack(data: np.ndarray, n: int, point_step: int, off_x: int, off_y: int, off_z: int, off_i: int) -> np.ndarray:
    """a1: PointCloud2 bytes -> (n, 4) float32 xyzi (subscribers at pc_preprocessing_main.cpp:520-525)."""
    raw = np.frombuffer(np.ascontiguousarray(data).tobytes(), dtype=np.uint8)[: n * point_step].reshape(n, point_step)
    out = np.zeros((n, 4), dtype=F32)
    for k, off in enumerate((off_x, off_y, off_z, off_i)):
        if off < 0:
            continue
        out[:, k] = np.ascontiguousarray(raw[:, off:off + 4]).view("<f4")[:, 0]
    return out


def transform(xyzi: np.ndarray, m: np.ndarray, is_dense: bool = True) -> np.ndarray:
    """a2: pcl::transformPointCloud (PCL 1.8.1): x' = ((m00*x + m01*y) + m02*z) + m03, unfused, left to right.
    Reference call sites pc_preprocessing_main.cpp:322..465. m: 12 floats, row-major 3x4."""
    m = np.asarray(m, dtype=F32).reshape(3, 4)
    x, y, z = xyzi[:, 0].astype(F32), xyzi[:, 1].astype(F32), xyzi[:, 2].astype(F32)
    out = xyzi.astype(F32).copy()
    with np.errstate(invalid="ignore", over="ignore"):
        for r in range(3):
            out[:, r] = ((m[r, 0] * x + m[r, 1] * y) + m[r, 2] * z) + m[r, 3]
    if not is_dense:
        bad = ~(np.isfinite(x) & np.isfinite(y) & np.isfinite(z))
        out[bad, :3] = xyzi[bad, :3]
    return out


def passthrough_mask(xyzi: np.ndarray, axis: int, lo, hi, negative: bool = False) -> np.ndarray:
    """a3..a6: pcl::PassThrough::applyFilterIndices (PCL 1.8.1): float limits, inclusive, non-finite rejected.
    Reference getROI pc_preprocessing_main.cpp:20-40, getCloudPart :49-59. PCL's two tests, literally: a point is dropped
    when `v < lo || v > hi`, or with `negative` when `v >= lo && v <= hi` -- so a NaN limit drops nothing (every finite
    value is kept) in either form."""
    lo, hi = F32(lo), F32(hi)
    v = xyzi[:, axis]
    fin = np.isfinite(xyzi[:, 0]) & np.isfinite(xyzi[:, 1]) & np.isfinite(xyzi[:, 2]) & np.isfinite(v)
    with np.errstate(invalid="ignore"):
        drop = ((v >= lo) & (v <= hi)) if negative else ((v < lo) | (v > hi))
    return fin & ~drop


def crop(xyzi: np.ndarray, passes) -> np.ndarray:
    """Chained PassThrough = logical AND; returns the boolean keep mask. passes: iterable of (axis, lo, hi, negative)."""
    keep = np.ones(len(xyzi), dtype=bool)
    for (axis, lo, hi, negative) in passes:
        keep &= passthrough_mask(xyzi, axis, lo, hi, bool(negative))
    return keep


def voxelgrid(xyzi: np.ndarray, leaf, min_points: int = 0, downsample_all: bool = True, force64: bool = True,
              bounds=None):
    """a8: pcl::VoxelGrid::applyFilter (PCL 1.8.1), reference voxelgrid pc_preprocessing_main.cpp:168-177.

    Returns dict(idx, count, centroid_f64, point_idx, min_b, max_b, div_b, pcl_overflow). Centroids are accumulated in
    float64 in ascending point order (the tolerance anchor). bounds = (min_p, max_p) replaces the cloud's own bounding
    box (used for a cloud that is one part of a larger, partitioned cloud)."""
    xyzi = np.asarray(xyzi, dtype=F32)
    n = len(xyzi)
    leaf = np.asarray(leaf, dtype=F32)
    inv = (F32(1.0) / leaf).astype(F32)
    fin = np.isfinite(xyzi[:, 0]) & np.isfinite(xyzi[:, 1]) & np.isfinite(xyzi[:, 2])
    res = dict(idx=np.zeros(0, np.int64), count=np.zeros(0, np.uint32), centroid_f64=np.zeros((0, 4)),
               point_idx=np.full(n, -1, np.int64), min_b=np.zeros(3, np.int64), max_b=np.zeros(3, np.int64),
               div_b=np.zeros(3, np.int64), pcl_overflow=False)
    if not fin.any():
        return res
    pts = xyzi[fin]
    min_p = pts[:, :3].min(axis=0).astype(F32)
    max_p = pts[:, :3].max(axis=0).astype(F32)
    if bounds is not None:
        min_p = np.minimum(min_p, np.asarray(bounds[0], F32))
        max_p = np.maximum(max_p, np.asarray(bounds[1], F32))
    d = ((max_p - min_p).astype(F32) * inv).astype(F32)
    dxyz = [int(np.trunc(np.float64(v))) + 1 for v in d]
    res["pcl_overflow"] = (dxyz[0] * dxyz[1] * dxyz[2]) > INT32_MAX
    min_b = np.floor((min_p * inv).astype(F32)).astype(np.int64)
    max_b = np.floor((max_p * inv).astype(F32)).astype(np.int64)
    div_b = max_b - min_b + 1
    res.update(min_b=min_b, max_b=max_b, div_b=div_b)
    if res["pcl_overflow"] and not force64:
        return res
    cell = np.floor((pts[:, :3] * inv[None, :]).astype(F32)).astype(np.int64) - min_b[None, :]
    idx = cell[:, 0] + cell[:, 1] * div_b[0] + cell[:, 2] * div_b[0] * div_b[1]
    pidx = np.full(n, -1, np.int64)
    pidx[fin] = idx
    res["point_idx"] = pidx
    order = np.argsort(idx, kind="stable")
    sidx = idx[order]
    uniq, start, cnt = np.unique(sidx, return_index=True, return_counts=True)
    keep = cnt >= max(int(min_points), 0)
    sums = np.add.reduceat(pts[order].astype(np.float64), start, axis=0) if len(start) else np.zeros((0, 4))
    cent = sums / cnt[:, None]
    if not downsample_all:
        cent[:, 3] = 0.0
    res.update(idx=uniq[keep], count=cnt[keep].astype(np.uint32), centroid_f64=cent[keep])
    return res


def tf_to_matrix(quat_xyzw, origin_xyz) -> np.ndarray:
    """Eigen 3.3.4 Quaternionf::toRotationMatrix + translation, as pcl_ros builds the Affine3f from a tf::Transform."""
    x, y, z, w = (F32(v) for v in quat_xyzw)
    tx, ty, tz = F32(2) * x, F32(2) * y, F32(2) * z
    twx, twy, twz = tx * w, ty * w, tz * w
    txx, txy, txz = tx * x, ty * x, tz * x
    tyy, tyz, tzz = ty * y, tz * y, tz * z
    one = F32(1)
    return np.array([
        one - (tyy + tzz), txy - twz, txz + twy, F32(origin_xyz[0]),
        txy + twz, one - (txx + tzz), tyz - twx, F32(origin_xyz[1]),
        txz - twy, tyz + twx, one - (txx + tyy), F32(origin_xyz[2])], dtype=F32)


def merge_frame(clouds, passes, leaf, min_points=0, downsample_all=True, force64=True):
    """Whole path: per sensor unpack -> transform -> crop; concat in sensor order; VoxelGrid.
    clouds: list of dict(data, n_points, point_step, off_x, off_y, off_z, off_i, is_dense, m).
    Returns dict(survivor_xyzi, survivor_src, voxel=<voxelgrid dict>)."""
    surv, src, base = [], [], 0
    for c in clouds:
        p = unpack(c["data"], c["n_points"], c["point_step"], c["off_x"], c["off_y"], c["off_z"], c["off_i"])
        t = transform(p, c["m"], bool(c["is_dense"]))
        keep = crop(t, passes) if len(passes) else np.ones(len(t), dtype=bool)
        surv.append(t[keep])
        src.append(base + np.nonzero(keep)[0])
        base += c["n_points"]
    sx = np.concatenate(surv) if surv else np.zeros((0, 4), F32)
    ss = np.concatenate(src).astype(np.uint32) if src else np.zeros(0, np.uint32)
    return dict(survivor_xyzi=sx, survivor_src=ss, voxel=voxelgrid(sx, leaf, min_points, downsample_all, force64))


# ---- RANSAC ground plane (pcl::SACSegmentation, SACMODEL_PLANE + SAC_RANSAC; pc_preprocessing_main.cpp:95-108) ------------
def _sum4(l0, l1, l2, l3, order: int):
    """Eigen's 4-wide float reduction: 0 = SSE2 (l0+l2)+(l1+l3), 1 = SSE3 (l0+l1)+(l2+l3), 2 = scalar ((l0+l1)+l2)+l3."""
    l0, l1, l2, l3 = (np.asarray(v, F32) for v in (l0, l1, l2, l3))
    if order == 0:
        return ((l0 + l2).astype(F32) + (l1 + l3).astype(F32)).astype(F32)
    if order == 1:
        return ((l0 + l1).astype(F32) + (l2 + l3).astype(F32)).astype(F32)
    return (((l0 + l1).astype(F32) + l2).astype(F32) + l3).astype(F32)


def plane_of_sample(p0, p1, p2, order: int = 0):
    """isSampleGood + computeModelCoefficients of SampleConsensusModelPlane: (good, coefficients[4] float32)."""
    p0, p1, p2 = (np.asarray(v, F32)[:3] for v in (p0, p1, p2))
    with np.errstate(all="ignore"):
        u = (p1 - p0).astype(F32)
        v = (p2 - p0).astype(F32)
        q = (u / v).astype(F32)
        good = bool(q[0] != q[1]) or bool(q[2] != q[1])
        c = np.zeros(4, F32)
        c[0] = F32(F32(u[1] * v[2]) - F32(u[2] * v[1]))
        c[1] = F32(F32(u[2] * v[0]) - F32(u[0] * v[2]))
        c[2] = F32(F32(u[0] * v[1]) - F32(u[1] * v[0]))
        z = _sum4(c[0] * c[0], c[1] * c[1], c[2] * c[2], c[3] * c[3], order)
        if z > 0:
            c = (c / np.sqrt(z, dtype=F32)).astype(F32)
        c[3] = F32(-1.0) * _sum4(c[0] * p0[0], c[1] * p0[1], c[2] * p0[2], c[3] * F32(1.0), order)
    return good, c


def plane_inlier_mask(xyzi: np.ndarray, c: np.ndarray, threshold: float, order: int = 0) -> np.ndarray:
    """countWithinDistance / selectWithinDistance: |dot(c, (x, y, z, 1))| < threshold (float distance, double threshold)."""
    x = np.asarray(xyzi, F32)
    with np.errstate(all="ignore"):
        d = np.abs(_sum4(c[0] * x[:, 0], c[1] * x[:, 1], c[2] * x[:, 2], np.broadcast_to(c[3], x[:, 0].shape), order))
        return d.astype(np.float64) < float(threshold)


def plane_ransac(xyzi: np.ndarray, threshold: float, probability: float = 0.99, max_iterations: int = 1000,
                 seed: int = 12345, order: int = 0) -> dict:
    """RandomSampleConsensus::computeModel with PCL's sampler (mt19937(seed) >> 1, partial shuffle); no refit."""
    x = np.ascontiguousarray(xyzi, F32).reshape(-1, 4)
    n = len(x)
    out = {"found": False, "iterations": 0, "draws": 0, "best_count": 0, "sample": np.full(3, -1, np.int32), "coeff": np.zeros(4, F32)}
    if n < 3:
        return out
    raw = np.random.RandomState(seed)._bit_generator  # init_genrand(seed), as boost::mt19937::seed(value)
    shuffled = np.arange(n, dtype=np.int64)
    iterations, draws, best, k = 0, 0, -INT32_MAX, 1.0
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
            good, c = plane_of_sample(x[sel[0]], x[sel[1]], x[sel[2]], order)
            if good:
                got = True
                break
        if not got:
            break
        cnt = int(plane_inlier_mask(x, c, threshold, order).sum())
        if cnt > best:
            best = cnt
            out.update(found=True, best_count=cnt, sample=sel.astype(np.int32), coeff=c.copy())
            w = best / n
            p_no = 1.0 - w ** 3.0
            p_no = min(max(np.finfo(np.float64).eps, p_no), 1.0 - np.finfo(np.float64).eps)
            k = log_p / np.log(p_no)
        iterations += 1
        if iterations > max_iterations:
            break
    out.update(iterations=iterations, draws=draws)
    return out
