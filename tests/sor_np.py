"""numpy restatement of pcl::StatisticalOutlierRemoval (PCL 1.8.1 filters/impl/statistical_outlier_removal.hpp,
applyFilterIndices) -- TEST INFRASTRUCTURE ONLY, independent of tests/sor_oracle.cpp:

  1. the mean_k + 1 smallest float32 squared distances of every finite point to the finite points of its cloud (itself
     included), in FLANN's L2_Simple order (dx*dx + dy*dy) + dz*dz;
  2. dist_sum (double, from 0) += sqrt(nn[k]) for k = 1 .. mean_k ascending -- sqrt of the float (sqrt_mode 0) or of the
     promoted double (1) --, distance = (float)(dist_sum / mean_k); a non-finite point gets 0 and is not valid;
  3. sum += d and sq_sum += d * d (a float product) over ALL points in index order (doubles), mean = sum / valid,
     variance = (sq_sum - sum * sum / valid) / (valid - 1), stddev = sqrt(variance), threshold = mean + std_mul * stddev;
  4. removed iff (double)d > threshold (negative: <=).
A cloud with 0 < valid <= mean_k (PCL reads past its neighbour vectors) keeps every point; its distances are 0.

Candidates come from scipy's cKDTree with slack; the float32 distances are recomputed here, and the slack is checked to
have sufficed: every point the tree did not return is at least as far (float squared distance, with rounding margin) as
the mean_k + 1-th value kept. Where it was not, the query is repeated with more candidates."""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

F32 = np.float32


def _sq_dist(q, c):
    """float32 squared distances of q [m,3] to c [m,k,3] in FLANN's order, never fused."""
    dx = (q[:, None, 0] - c[:, :, 0]).astype(F32)
    dy = (q[:, None, 1] - c[:, :, 1]).astype(F32)
    dz = (q[:, None, 2] - c[:, :, 2]).astype(F32)
    return ((dx * dx + dy * dy).astype(F32) + (dz * dz).astype(F32)).astype(F32)


def knn_sq(xyz: np.ndarray, kp1: int, chunk: int = 65536, workers: int = -1) -> np.ndarray:
    """[n, kp1] ascending float32 squared distances of every point of xyz (finite, float32) to the kp1 nearest."""
    n = len(xyz)
    tree = cKDTree(xyz.astype(np.float64))
    out = np.empty((n, kp1), F32)
    for a in range(0, n, chunk):
        q = xyz[a:a + chunk]
        todo = np.arange(len(q))
        k = min(n, kp1 + 8)
        while len(todo):
            dd, ii = tree.query(q[todo].astype(np.float64), k=k, workers=workers)
            dd = dd.reshape(len(todo), -1)
            ii = ii.reshape(len(todo), -1)
            f = np.sort(_sq_dist(q[todo], xyz[ii]), axis=1)[:, :kp1]
            if k >= n:
                ok = np.ones(len(todo), bool)
            else:
                # a point the tree did not return is >= dd[:, -1] away (exactly); its float squared distance is then
                # >= dd^2 (1 - 2^-21) -- the float rounding of the three subtractions, squares and sums is below that
                far = (dd[:, -1] ** 2) * (1.0 - 2.0 ** -21)
                ok = f[:, -1].astype(np.float64) <= far
            out[a + todo[ok]] = f[ok]
            todo = todo[~ok]
            k = min(n, 2 * k)
    return out


def serial_sum(v: np.ndarray) -> float:
    """sum in index order with a double accumulator (ufunc.accumulate is sequential, unlike sum())."""
    return float(np.add.accumulate(np.concatenate([[0.0], v.astype(np.float64)]))[-1])


def sor_cloud(xyzi: np.ndarray, mean_k: int, std_mul: float, negative: bool = False, sqrt_mode: int = 0,
              workers: int = -1) -> dict:
    a = np.asarray(xyzi, F32).reshape(-1, 4)
    n = len(a)
    fin = np.isfinite(a[:, :3]).all(1)
    valid = int(fin.sum())
    dist = np.zeros(n, F32)
    too_few = 0 < valid <= mean_k
    if valid and not too_few:
        nn = knn_sq(np.ascontiguousarray(a[fin, :3]), mean_k + 1, workers=workers)
        s = np.zeros(valid, np.float64)
        for k in range(1, mean_k + 1):  # ascending, one column at a time: the order of PCL's loop
            col = nn[:, k]
            s = s + (np.sqrt(col).astype(np.float64) if sqrt_mode == 0 else np.sqrt(col.astype(np.float64)))
        dist[fin] = (s / mean_k).astype(F32)
    sm = np.float64(serial_sum(dist))
    sq = np.float64(serial_sum((dist * dist).astype(F32)))
    vd = np.float64(valid)
    with np.errstate(all="ignore"):  # IEEE doubles: 0 / 0 is NaN here as in PCL
        mean = sm / vd
        variance = (sq - sm * sm / vd) / (vd - 1.0)
        stddev = np.sqrt(variance)
        threshold = mean + np.float64(std_mul) * stddev
    d64 = dist.astype(np.float64)
    with np.errstate(invalid="ignore"):
        removed = (d64 <= threshold) if negative else (d64 > threshold)
    if too_few:
        removed[:] = False
    return {"distances": dist, "keep": ~removed, "mean": float(mean), "stddev": float(stddev),
            "threshold": float(threshold), "n_valid": valid, "too_few": too_few, "sum": float(sm), "sq_sum": float(sq)}


def sor(clouds, mean_k: int, std_mul: float, negative: bool = False, sqrt_mode: int = 0) -> list:
    return [sor_cloud(c, mean_k, std_mul, negative, sqrt_mode) for c in clouds]
