"""Input clouds of the Euclidean cluster extraction tests and benchmark (TEST INFRASTRUCTURE ONLY). (n, 4) float32 xyzi."""
from __future__ import annotations

import numpy as np

from sor_cases import blobs, fused_frame, lattice, roi_cloud, shell_faces, with_duplicates, with_nonfinite, zone_clouds  # noqa: F401
from ec_np import r2_of

F32 = np.float32


def _cloud(xyz) -> np.ndarray:
    xyz = np.asarray(xyz, F32).reshape(-1, 3)
    return np.ascontiguousarray(np.column_stack([xyz, np.arange(len(xyz), dtype=F32)]))


def ulp_pairs(seed: int, tolerance: float, k: int = 3, n: int = 400) -> np.ndarray:
    """chains of three points in random directions, each step sqrt(r2) shifted by -k .. +k ulps, 3 m apart: every step
    falls on either side of the strict < and joins or breaks its chain."""
    rng = np.random.default_rng(seed)
    step0 = F32(np.sqrt(np.float64(r2_of(tolerance))))
    pts = []
    for c in range(n):
        d = rng.normal(size=3)
        d /= np.linalg.norm(d)
        base = np.array([(c % 20) * 3.0, (c // 20) * 3.0, 0.0]) + rng.uniform(-0.5, 0.5, 3)
        p = base.astype(F32)
        pts.append(p)
        for _ in range(2):
            s = step0
            for _ in range(abs(u := int(rng.integers(-k, k + 1)))):
                s = np.nextafter(s, F32(np.inf if u > 0 else -np.inf))
            p = (p + (d * float(s)).astype(F32)).astype(F32)
            pts.append(p)
    return _cloud(np.array(pts))


def snake(seed: int, tolerance: float, n: int = 3000) -> np.ndarray:
    """two random walks of 0.9-tolerance steps winding through many cells, their points interleaved in index order."""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(2, n, 3))
    d /= np.linalg.norm(d, axis=2, keepdims=True)
    walks = np.cumsum(d * 0.9 * tolerance, axis=1) + np.array([[[0.0, 0.0, 0.0]], [[0.0, 0.0, 40.0 * tolerance]]])
    both = walks.reshape(-1, 3)
    return _cloud(both[rng.permutation(len(both))])


def equal_clusters(seed: int, n_clusters: int, size: int, tolerance: float, extra=()) -> np.ndarray:
    """n_clusters tight groups of `size` points (plus groups of the sizes in `extra`), 3 tolerances apart, shuffled."""
    rng = np.random.default_rng(seed)
    sizes = [size] * n_clusters + list(extra)
    side = int(np.ceil(np.sqrt(len(sizes))))
    pts = []
    for g, s in enumerate(sizes):
        c = np.array([(g % side) * 3.0 * tolerance, (g // side) * 3.0 * tolerance, 0.0])
        pts.append(c + rng.uniform(-0.2, 0.2, (s, 3)) * tolerance)
    xyz = np.concatenate(pts)
    return _cloud(xyz[rng.permutation(len(xyz))])


def dense_blob(seed: int, n: int = 100000, edge: float = 0.4) -> np.ndarray:
    """n points inside one cell of a 0.5 m tolerance: the m^2 walk of the hook kernel in its worst case."""
    rng = np.random.default_rng(seed)
    return _cloud(rng.uniform(0.0, edge, (n, 3)) + 0.55)
