"""Input clouds of the statistical outlier removal tests and benchmark (TEST INFRASTRUCTURE ONLY). (n, 4) float32 xyzi."""
from __future__ import annotations

import numpy as np

from cloud_merger_b200 import ROI_PASSES, synth

F32 = np.float32


def transformed(cloud, m):
    """sensor -> base in float32 (rows of the 3x4 extrinsic), intensity kept."""
    m = np.asarray(m, F32).reshape(-1)[:12].reshape(3, 4)
    out = np.empty_like(cloud)
    for r in range(3):
        out[:, r] = (cloud[:, 0] * m[r, 0] + cloud[:, 1] * m[r, 1] + cloud[:, 2] * m[r, 2] + m[r, 3]).astype(F32)
    out[:, 3] = cloud[:, 3]
    return out


def roi_cloud(seed: int, rings: int, az: int) -> np.ndarray:
    """a sensor cloud in the base frame, cropped to the ROI of getROI (64 x 2048: ~58 k points, 128 x 4096: ~233 k)."""
    cur = transformed(synth.lidar_cloud(seed, 0, 0, rings, az), synth.extrinsic(0, 4))
    for (axis, lo, hi, neg) in ROI_PASSES:
        v = cur[:, axis]
        cur = cur[(v >= F32(lo)) & (v <= F32(hi))]
    return np.ascontiguousarray(cur)


def fused_frame(seed: int, cfg: str = "cfg3") -> np.ndarray:
    """all sensor clouds of one frame, transformed and concatenated (cfg3: 8 x 256 k = 2 M points)."""
    clouds, mats = synth.frame_clouds(cfg, seed, 0)
    return np.ascontiguousarray(np.concatenate([transformed(c, m) for c, m in zip(clouds, mats)]))


def zone_clouds(cloud: np.ndarray, n: int = 5) -> list:
    """n consecutive x windows of a ROI cloud (the per-zone clouds of a proceedX)."""
    edges = np.linspace(-15.0, 60.0, n + 1)
    return [np.ascontiguousarray(cloud[(cloud[:, 0] >= edges[k]) & (cloud[:, 0] < edges[k + 1])]) for k in range(n)]


def blobs(seed: int, n: int, spread: float = 1.0, outliers: int = 20, far: float = 50.0) -> np.ndarray:
    """gaussian clusters plus a few far outliers (many cells away: many growth steps of the search)."""
    rng = np.random.default_rng(seed)
    centres = rng.uniform(-10, 10, (8, 3))
    pts = centres[rng.integers(0, 8, n)] + rng.normal(scale=spread, size=(n, 3))
    out = rng.normal(size=(outliers, 3))
    out = out / np.linalg.norm(out, axis=1, keepdims=True) * rng.uniform(far, 3 * far, (outliers, 1))
    xyz = np.concatenate([pts, out]).astype(F32)
    return np.ascontiguousarray(np.column_stack([xyz, rng.uniform(0, 100, len(xyz)).astype(F32)]))


def lattice(n_side: int, step: float = 0.25, origin=(0.0, 0.0, 0.0)) -> np.ndarray:
    """a cubic lattice: every point has 6 neighbours at one distance, 12 at the next -- ties at the k-th distance."""
    g = np.arange(n_side, dtype=F32) * F32(step)
    x, y, z = np.meshgrid(g, g, g, indexing="ij")
    xyz = np.column_stack([x.ravel(), y.ravel(), z.ravel()]).astype(F32) + np.asarray(origin, F32)
    return np.ascontiguousarray(np.column_stack([xyz, np.zeros(len(xyz), F32)]))


def with_duplicates(cloud: np.ndarray, seed: int, frac: float = 0.2) -> np.ndarray:
    rng = np.random.default_rng(seed)
    extra = cloud[rng.integers(0, len(cloud), int(frac * len(cloud)))]
    out = np.concatenate([cloud, extra])
    return np.ascontiguousarray(out[rng.permutation(len(out))])


def with_nonfinite(cloud: np.ndarray, seed: int, frac: float = 0.05) -> np.ndarray:
    rng = np.random.default_rng(seed)
    out = cloud.copy()
    rows = rng.choice(len(out), max(1, int(frac * len(out))), replace=False)
    vals = np.array([np.nan, np.inf, -np.inf], F32)
    for k, r in enumerate(rows):
        out[r, k % 3] = vals[k % 3]
    return out


def shell_faces(seed: int, cell: float, n: int = 600) -> np.ndarray:
    """pairs of points whose coordinates sit on multiples of `cell` (cell faces of the grid a forced edge makes) and one
    ulp either side, so neighbours fall just inside and just outside the cubes the search visits."""
    rng = np.random.default_rng(seed)
    base = (rng.integers(-20, 20, (n, 3)) * cell).astype(F32)
    ulps = rng.integers(-2, 3, (n, 3))
    xyz = base.copy()
    for a in range(3):
        for u in (-1, 1):
            sel = ulps[:, a] * u > 0
            for _ in range(2):
                xyz[sel, a] = np.nextafter(xyz[sel, a], F32(u * np.inf))
    jitter = (base + rng.uniform(-0.6, 0.6, (n, 3)).astype(F32) * F32(cell)).astype(F32)
    pts = np.concatenate([xyz, base, jitter]).astype(F32)
    return np.ascontiguousarray(np.column_stack([pts, np.zeros(len(pts), F32)]))
