"""numpy/scipy statement of pcl::NormalEstimation with a radius search (TEST INFRASTRUCTURE ONLY), independent of the C++
statement: candidates from a cKDTree ball query with slack, FLANN's float32 squared distance recomputed in its operation
order, the neighbour lists ordered by (d2, index) with lexsort, the nine running sums column by column in float32 (every
neighbourhood padded with zero terms, which leave a sum that started at +0 unchanged), and solve(): PCL 1.8.1's
computeMeanAndCovarianceMatrix / eigen33 / solvePlaneParameters / flipNormalTowardsViewpoint restated step by step in
numpy float32 scalars from PCL's source. Only the trig rule comes from cm_ne_math.h (through ctypes): it is stated
nowhere else."""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

import ne_oracle as O

F32 = np.float32


def neighbour_lists(xyzi, radius: float):
    """(order, starts): the neighbours of every point in FLANN's order, concatenated; starts[i] .. starts[i+1]."""
    a = np.asarray(xyzi, F32).reshape(-1, 4)
    n = len(a)
    fin = np.nonzero(np.isfinite(a[:, :3]).all(axis=1))[0]
    r2 = F32(float(radius) * float(radius))
    lists = [np.zeros(0, np.int64)] * n
    if len(fin):
        tree = cKDTree(a[fin, :3].astype(np.float64))
        slack = float(radius) * (1 + 1e-5) + 1e-30
        cand = tree.query_ball_point(a[fin, :3].astype(np.float64), slack)
        for q, c in zip(fin, cand):
            j = fin[np.asarray(c, np.int64)]
            d = a[j, :3] - a[q, :3]
            d2 = ((d[:, 0] * d[:, 0]).astype(F32) + (d[:, 1] * d[:, 1]).astype(F32)).astype(F32)
            d2 = (d2 + (d[:, 2] * d[:, 2]).astype(F32)).astype(F32)
            keep = d2 < r2
            j, d2 = j[keep], d2[keep]
            lists[q] = j[np.lexsort((j, d2))]
    return lists


def check_slack(xyzi, radius: float, lists, sample: int = 300, seed: int = 0) -> None:
    """The ball query's slack misses nothing: for a sample of queries, every finite point of the whole cloud with float
    d2 < r2 (brute force, FLANN's operation order) is in the list, and nothing else is."""
    a = np.asarray(xyzi, F32).reshape(-1, 4)
    fin = np.nonzero(np.isfinite(a[:, :3]).all(axis=1))[0]
    r2 = F32(float(radius) * float(radius))
    rng = np.random.default_rng(seed)
    for q in rng.choice(fin, min(sample, len(fin)), replace=False) if len(fin) else []:
        d = a[fin, :3] - a[q, :3]
        d2 = ((d[:, 0] * d[:, 0]).astype(F32) + (d[:, 1] * d[:, 1]).astype(F32)).astype(F32)
        d2 = (d2 + (d[:, 2] * d[:, 2]).astype(F32)).astype(F32)
        assert np.array_equal(np.sort(fin[d2 < r2]), np.sort(lists[q])), q


def _roots2(b, c):
    """pcl::computeRoots2: the literal 4.0 makes 4.0 * c and the difference double"""
    d = F32(float(F32(b * b)) - 4.0 * float(c))
    if d < 0.0:
        d = F32(0.0)
    sd = np.sqrt(d)
    return [F32(0.0), F32(F32(0.5) * F32(b - sd)), F32(F32(0.5) * F32(b + sd))]


def _roots3(m, path):
    """pcl::computeRoots on the scaled matrix m (3x3 of float32 scalars); path collects the branches taken"""
    m00, m01, m02, m11, m12, m22 = m[0][0], m[0][1], m[0][2], m[1][1], m[1][2], m[2][2]
    c0 = m00 * m11 * m22 + F32(2) * m01 * m02 * m12 - m00 * m12 * m12 - m11 * m02 * m02 - m22 * m01 * m01
    c1 = m00 * m11 - m01 * m01 + m00 * m22 - m02 * m02 + m11 * m22 - m12 * m12
    c2 = m00 + m11 + m22
    if abs(c0) < np.finfo(F32).eps:
        path.add("roots2")
        return _roots2(c2, c1)
    path.add("trig")
    s_inv3, s_sqrt3 = F32(1.0 / 3.0), np.sqrt(F32(3.0))
    c2_over_3 = c2 * s_inv3
    a_over_3 = (c1 - c2 * c2_over_3) * s_inv3
    if a_over_3 > F32(0):
        a_over_3 = F32(0)
    half_b = F32(0.5) * (c0 + c2_over_3 * (F32(2) * c2_over_3 * c2_over_3 - c1))
    q = half_b * half_b + a_over_3 * a_over_3 * a_over_3
    if q > F32(0):
        q = F32(0)
    rho = np.sqrt(-a_over_3)
    theta = O.atan2(np.sqrt(-q), half_b) * s_inv3
    cos_t, sin_t = O.cos(theta), O.sin(theta)
    r = [c2_over_3 + F32(2) * rho * cos_t, c2_over_3 - rho * (cos_t + s_sqrt3 * sin_t),
         c2_over_3 - rho * (cos_t - s_sqrt3 * sin_t)]
    if r[0] >= r[1]:
        r[0], r[1] = r[1], r[0]
    if r[1] >= r[2]:
        r[1], r[2] = r[2], r[1]
        if r[0] >= r[1]:
            r[0], r[1] = r[1], r[0]
    if r[0] <= 0:
        path.add("root0_neg")
        return _roots2(c2, c1)
    return r


def _cross(u, v):
    return [u[1] * v[2] - u[2] * v[1], u[2] * v[0] - u[0] * v[2], u[0] * v[1] - u[1] * v[0]]


def solve(sums, count: int, p, viewpoint, norm_order: str = "eigen", flip_order: str = "pcl", path=None):
    """nx ny nz curvature of one neighbourhood from its nine float32 running sums, as PCL 1.8.1 computes them.
    norm_order: "eigen" = Eigen 3.3's a0 + (a1 + a2) for squaredNorm, "left" = (a0 + a1) + a2. flip_order: "pcl" = the
    float& flipNormalTowardsViewpoint's (vx*nx + vy*ny) + vz*nz, "eigen" = a dot's a0 + (a1 + a2)."""
    path = set() if path is None else path
    nan = np.array(0x7FC00000, np.uint32).view(F32)
    with np.errstate(all="ignore"):
        acc = [F32(v) for v in sums]
        cnt = F32(count)
        acc = [a / cnt for a in acc]
        cov = np.empty((3, 3), F32)
        cov[0, 0] = acc[0] - acc[6] * acc[6]
        cov[0, 1] = acc[1] - acc[6] * acc[7]
        cov[0, 2] = acc[2] - acc[6] * acc[8]
        cov[1, 1] = acc[3] - acc[7] * acc[7]
        cov[1, 2] = acc[4] - acc[7] * acc[8]
        cov[2, 2] = acc[5] - acc[8] * acc[8]
        cov[1, 0], cov[2, 0], cov[2, 1] = cov[0, 1], cov[0, 2], cov[1, 2]
        if not np.isfinite(cov).all():  # documented deviation
            return [nan] * 4
        scale = np.abs(cov).max()
        if scale <= np.finfo(F32).tiny:
            scale = F32(1.0)
        m = [[cov[i, j] / scale for j in range(3)] for i in range(3)]
        r = _roots3(m, path)
        eigenvalue = r[0] * scale
        for i in range(3):
            m[i][i] = m[i][i] - r[0]
        vecs = [_cross(m[0], m[1]), _cross(m[0], m[2]), _cross(m[1], m[2])]
        sq = [[v[0] * v[0], v[1] * v[1], v[2] * v[2]] for v in vecs]
        lens = [a[0] + (a[1] + a[2]) if norm_order == "eigen" else (a[0] + a[1]) + a[2] for a in sq]
        if lens[0] >= lens[1] and lens[0] >= lens[2]:
            k = 0
        elif lens[1] >= lens[0] and lens[1] >= lens[2]:
            k = 1
        else:
            k = 2
        path.add("pick%d" % (k + 1))
        nrm = np.sqrt(lens[k])
        n = [vecs[k][i] / nrm for i in range(3)]
        eig_sum = cov[0, 0] + cov[1, 1] + cov[2, 2]
        curvature = abs(eigenvalue / eig_sum) if eig_sum != 0 else F32(0)
        d = [F32(viewpoint[i]) - F32(p[i]) for i in range(3)]
        t = [d[i] * n[i] for i in range(3)]
        cos_theta = (t[0] + t[1]) + t[2] if flip_order == "pcl" else t[0] + (t[1] + t[2])
        if cos_theta < 0:
            n = [v * F32(-1) for v in n]
            path.add("flip")
    out = [F32(v) for v in n] + [F32(curvature)]
    return [nan if np.isnan(v) else v for v in out]


def sums_of(xyzi, radius: float):
    """(sums [n, 9] float32, counts [n]): the nine running sums of every point's neighbourhood in FLANN's order"""
    a = np.ascontiguousarray(np.asarray(xyzi, F32).reshape(-1, 4))
    lists = neighbour_lists(a, radius)
    n = len(a)
    counts = np.array([len(x) for x in lists], np.int64)
    L = int(counts.max()) if n else 0
    idx = np.full((n, max(L, 1)), -1, np.int64)
    for i, x in enumerate(lists):
        idx[i, :len(x)] = x
    xyz = np.concatenate([a[:, :3], np.zeros((1, 3), F32)])  # row n: the zero padding
    cols = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]
    sums = np.zeros((n, 9), F32)
    for k in range(L):
        p = xyz[np.where(idx[:, k] >= 0, idx[:, k], n)]
        for c, (u, v) in enumerate(cols):
            sums[:, c] = (sums[:, c] + (p[:, u] * p[:, v]).astype(F32)).astype(F32)
        for c in range(3):
            sums[:, 6 + c] = (sums[:, 6 + c] + p[:, c]).astype(F32)
    return sums, counts


def normals(xyzi, radius: float, viewpoint=(0.0, 0.0, 0.0)) -> np.ndarray:
    a = np.ascontiguousarray(np.asarray(xyzi, F32).reshape(-1, 4))
    n = len(a)
    sums, counts = sums_of(a, radius)
    nan = np.array(0x7FC00000, np.uint32).view(F32)
    out = np.full((n, 4), nan, F32)
    for i in range(n):
        if counts[i] >= 3 and np.isfinite(a[i, :3]).all():
            out[i] = solve(sums[i], int(counts[i]), a[i, :3], viewpoint)
    return out
