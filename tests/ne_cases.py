"""Input clouds of the normal estimation tests and benchmark (TEST INFRASTRUCTURE ONLY). (n, 4) float32 xyzi."""
from __future__ import annotations

import numpy as np

from sor_cases import blobs, fused_frame, lattice, roi_cloud, shell_faces, with_duplicates, with_nonfinite, zone_clouds  # noqa: F401

F32 = np.float32


def cloud(xyz) -> np.ndarray:
    xyz = np.asarray(xyz, F32).reshape(-1, 3)
    return np.ascontiguousarray(np.column_stack([xyz, np.arange(len(xyz), dtype=F32)]))


def r2_of(radius: float) -> np.float32:
    """KdTreeFLANN::radiusSearch of NormalEstimation: (float)(radius * radius), the double square narrowed."""
    return F32(float(radius) * float(radius))


def ulp_edges(seed: int, radius: float, k: int = 2, n: int = 300) -> np.ndarray:
    """groups 3 m apart: a query, three points around it at 0.3 radius and one at sqrt(r2) shifted by -k .. +k ulps in a
    random direction, so that one neighbour falls on either side of the strict < and changes the normal."""
    rng = np.random.default_rng(seed)
    step0 = F32(np.sqrt(np.float64(r2_of(radius))))
    pts = []
    for c in range(n):
        base = (np.array([(c % 20) * 3.0, (c // 20) * 3.0, 0.0]) + rng.uniform(-0.5, 0.5, 3)).astype(F32)
        pts.append(base)
        for _ in range(3):
            pts.append((base + rng.normal(size=3) * 0.3 * radius).astype(F32))
        d = rng.normal(size=3)
        d /= np.linalg.norm(d)
        s = step0
        u = int(rng.integers(-k, k + 1))
        for _ in range(abs(u)):
            s = np.nextafter(s, F32(np.inf if u > 0 else -np.inf))
        pts.append((base + (d * float(s)).astype(F32)).astype(F32))
    return cloud(np.array(pts))


def ball(seed: int, n: int, centre, r: float) -> np.ndarray:
    """n points uniform in a ball of radius r (xyz only)."""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return (np.asarray(centre) + d * r * rng.uniform(0, 1, (n, 1)) ** (1 / 3)).astype(F32)


def exact_neighbourhoods(sizes, radius: float, seed: int = 1) -> np.ndarray:
    """one tight group of every size (inside a ball of radius / 4: every member sees exactly the group), 4 radii apart,
    the groups' points interleaved in index order."""
    parts = [ball(seed + k, s, (k * 4.0 * radius, 0.0, 0.0), radius / 4) for k, s in enumerate(sizes)]
    xyz = np.concatenate(parts)
    return cloud(xyz[np.random.default_rng(seed).permutation(len(xyz))])


def dense_blob(seed: int, n: int, radius: float) -> np.ndarray:
    """n points within one radius of each other (a cube of edge radius / 2): every query sees the whole cloud."""
    rng = np.random.default_rng(seed)
    return cloud(rng.uniform(0.0, radius / 2, (n, 3)) + 0.55)


def small_groups(radius: float) -> np.ndarray:
    """isolated groups of 1, 2, 3 and 4 points (neighbourhoods below and at PCL's minimum of 3), a line of 3 (a
    singular covariance), three exact duplicates (a zero covariance: NaN normal, curvature 0)."""
    pts = []
    for g, m in enumerate((1, 2, 3, 4)):
        for j in range(m):
            pts.append((g * 10.0 + 0.1 * radius * j, 0.05 * radius * (j % 2), 0.03 * radius * (j // 2)))
    pts += [(50.0 + 0.2 * radius * j, 0.0, 0.0) for j in range(3)]
    pts += [(60.0, 1.0, 2.0)] * 3
    return cloud(np.array(pts))


def eigen_family(seed: int, radius: float) -> np.ndarray:
    """groups 5 radii apart built for the branches of pcl::eigen33: exact planes (z = 0, y = c, x = c: |c0| < eps and
    each of the three cross-product picks), planes far from the origin (roots[0] <= 0 after the closed form), noisy
    blobs (the trig path), rotationally symmetric sets (two equal eigenvalues: the q clamp and the -0 branch), lines."""
    rng = np.random.default_rng(seed)
    groups = []
    r = radius * 0.3
    for k in range(12):
        u, v = rng.uniform(-r, r, (2, 9))
        groups.append(np.column_stack([u, v, np.zeros(9)]))          # normal z
        groups.append(np.column_stack([u, np.full(9, 0.25 * r), v]))  # normal y
        groups.append(np.column_stack([np.full(9, -0.5 * r), u, v]))  # normal x
        w = rng.normal(size=(12, 3)) * r * np.array([1.0, 0.6, 0.2])
        groups.append(w)                                              # a generic blob
        a = np.linspace(0, 2 * np.pi, 8, endpoint=False) + rng.uniform(0, 1)
        ring = np.column_stack([np.cos(a), np.sin(a), np.zeros(8)]) * r
        groups.append(np.concatenate([ring, [[0, 0, 0.3 * r], [0, 0, -0.3 * r]]]))   # xx = yy
        groups.append(np.concatenate([ring, [[0, 0, 0.7071 * r], [0, 0, -0.7071 * r]]]))  # nearly isotropic
        t = rng.uniform(-r, r, 6)
        groups.append(np.column_stack([t, 0.5 * t, -0.25 * t]))        # a line
        groups.append(np.column_stack([u, v, 1e-4 * r * rng.normal(size=9)]))  # nearly planar
    out = []
    for g, pts in enumerate(groups):
        out.append(pts + np.array([(g % 16) * 5.0 * radius, (g // 16) * 5.0 * radius, 0.0]))
    far = np.column_stack([rng.uniform(-r, r, (40, 2)), np.zeros(40)]) + np.array([1000.0, 2000.0, 300.0])
    far = np.concatenate([far[k * 8:(k + 1) * 8] + np.array([k * 5.0 * radius, 0, 0]) for k in range(5)])
    return cloud(np.concatenate(out + [far]))


def flip_ties(seed: int, count: int = 6, radius: float = 1.0) -> list:
    """(cloud, viewpoint) pairs: a noisy planar patch and a viewpoint near the tangent plane of its point 0, where
    flipNormalTowardsViewpoint's (vx*nx + vy*ny) + vz*nz and Eigen's a0 + (a1 + a2) decide the flip differently."""
    import ne_np as NP
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < count:
        m = int(rng.integers(5, 30))
        xyz = (rng.normal(size=(m, 3)) * np.array([0.2, 0.15, 0.01]) @ np.linalg.qr(rng.normal(size=(3, 3)))[0]
               + rng.uniform(-20, 20, 3)).astype(F32)
        c = cloud(xyz)
        sums, counts = NP.sums_of(c, radius)
        q = c[0, :3]
        n = np.array(NP.solve(sums[0], int(counts[0]), q, (0, 0, 0))[:3], F32)
        if not np.isfinite(n).all() or (np.abs(n) < 1e-3).any():
            continue
        for _ in range(60):
            t = F32(rng.uniform(0.5, 4.0))
            d = np.array([t / n[0], -t / n[1], F32(rng.uniform(-1, 1)) * F32(2.0 ** -rng.integers(18, 30)) / n[2]], F32)
            vp = (q + d).astype(F32)
            a = NP.solve(sums[0], int(counts[0]), q, vp, flip_order="pcl")
            b = NP.solve(sums[0], int(counts[0]), q, vp, flip_order="eigen")
            if np.array(a, F32).view(np.uint32).tolist() != np.array(b, F32).view(np.uint32).tolist():
                out.append((c, tuple(float(v) for v in vp)))
                break
    return out
