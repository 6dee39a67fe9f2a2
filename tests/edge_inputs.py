"""Seeded edge-case inputs for the voxel and crop kernels (tests only).

Random clouds almost never put a coordinate where the float32 formulas are fragile. These generators do so on purpose:

  A  lattice points: coordinates on and a few ulps around the voxel planes k * leaf, where floor(f32(x * inv)) decides the
     cell and a kernel that divided, fused or rounded the product differently would pick the neighbour cell;
  B  crop-limit points: transformed coordinates exactly on a PassThrough / box limit and one ulp either side, -0.0 against
     a limit of 0.0, subnormal coordinates and intensities;
  C  large offsets: map-frame clouds kilometres from the origin (coarsest float32 cells and centroid sums);
  D  grid-size boundaries: clouds whose extent puts the cell count, the key width or PCL's INT32 guard exactly on or one
     cell past a threshold.

Every generator is deterministic in its seed and returns (n, 4) float32 xyzi rows.
"""
from __future__ import annotations

import numpy as np

F32 = np.float32
LEAVES = (0.1, 0.05, 0.035, 1.0 / 3.0, 0.25, 1.0)
ULPS = (1, 2, 3)


def inv_of(leaf) -> np.float32:
    """1 / leaf as pcl::VoxelGrid computes it: a float32 division of float32 values."""
    return F32(F32(1.0) / F32(leaf))


def step_ulps(x, k: int):
    """x moved by k float32 ulps (k < 0: towards -inf)."""
    x = np.asarray(x, F32)
    to = F32(np.inf) if k > 0 else F32(-np.inf)
    for _ in range(abs(k)):
        x = np.nextafter(x, to).astype(F32)
    return x


def lattice_values(leaf, ks) -> np.ndarray:
    """x0 = f32(k * leaf) for every k and its +-1, +-2, +-3 ulp neighbours (float32, 7 values per k)."""
    x0 = (np.asarray(ks, np.float64) * float(F32(leaf))).astype(F32)
    vals = [x0] + [step_ulps(x0, s * u) for u in ULPS for s in (1, -1)]
    return np.concatenate(vals)


def _filler(rng, n, lo, hi):
    p = np.empty((n, 4), F32)
    p[:, :3] = rng.uniform(lo, hi, size=(n, 3)).astype(F32)
    p[:, 3] = rng.uniform(0.0, 255.0, size=n).astype(F32)
    return p


def lattice_cloud(seed: int, leaf, n_lattice: int = 20000, n_filler: int = 20000, k_span: int = 60,
                  centre=(0.0, 0.0, 0.0)) -> np.ndarray:
    """Family A (and, with a far centre, family C): points whose every coordinate lies on or within 3 ulps of a voxel plane
    around `centre` (negative, zero and positive cells when the centre is the origin), mixed into uniform filler points."""
    rng = np.random.default_rng(seed)
    leaf = float(F32(leaf))
    axes = []
    for a in range(3):
        k0 = int(np.floor(centre[a] / leaf))
        vals = lattice_values(leaf, np.arange(k0 - k_span, k0 + k_span + 1))
        axes.append(vals[rng.integers(0, len(vals), size=n_lattice)])
    lat = np.empty((n_lattice, 4), F32)
    lat[:, 0], lat[:, 1], lat[:, 2] = axes
    lat[:, 3] = rng.uniform(0.0, 255.0, size=n_lattice).astype(F32)
    c = np.asarray(centre, np.float64)
    fill = _filler(rng, n_filler, -k_span * leaf, k_span * leaf)
    fill[:, :3] = (fill[:, :3].astype(np.float64) + c).astype(F32)
    out = np.concatenate([lat, fill])
    return out[rng.permutation(len(out))]


def lattice_discrimination(leaf, x) -> dict:
    """Share of the coordinates x whose PCL cell floor(f32(x * inv)) differs from the exact floor(x / leaf) of the float64
    quotient, or from the cell of the product rounded towards zero: a kernel with either formula misplaces these points."""
    x = np.asarray(x, F32).reshape(-1)
    inv = inv_of(leaf)
    prod64 = x.astype(np.float64) * np.float64(inv)        # exact: a float32 product fits a float64
    rn = prod64.astype(F32)
    rz = np.where(np.abs(rn.astype(np.float64)) > np.abs(prod64), np.nextafter(rn, F32(0)), rn).astype(F32)
    cell = np.floor(rn)
    div = np.floor(x.astype(np.float64) / np.float64(F32(leaf)))
    return dict(vs_division=float(np.mean(cell != div)), vs_round_to_zero=float(np.mean(cell != np.floor(rz))),
                either=float(np.mean((cell != div) | (cell != np.floor(rz)))))


# ---- B: crop limits ----------------------------------------------------------------------------------------------------
def solve_translated(v, t) -> np.float32:
    """A float32 x with f32(x + t) == v exactly (unfused float addition, as the transform does), or None."""
    v, t = F32(v), F32(t)
    x0 = F32(np.float64(v) - np.float64(t))
    for k in range(-8, 9):
        x = step_ulps(x0, k)
        if F32(x + t) == v:
            return F32(x)
    return None


def limit_values(lo, hi):
    """lo and hi and one ulp either side of each."""
    lo, hi = F32(lo), F32(hi)
    return [step_ulps(lo, -1), lo, step_ulps(lo, 1), step_ulps(hi, -1), hi, step_ulps(hi, 1)]


def box_limit_cloud(seed: int, t, box, intensity_window=None, n_random: int = 3000) -> np.ndarray:
    """Family B for a sensor with identity rotation and translation t: for every axis and every limit value (lo, hi and one
    ulp either side) a group of points whose transformed coordinate is that value exactly, the other coordinates inside
    the box; with an intensity window, intensities on and one ulp around its limits too. Plus random points around the box."""
    rng = np.random.default_rng(seed)
    rows = []
    centre = [0.5 * (float(F32(lo)) + float(F32(hi))) for lo, hi in box]

    def inside(a):
        lo, hi = box[a]
        return F32(rng.uniform(float(F32(lo)) + 0.25 * (hi - lo), float(F32(hi)) - 0.25 * (hi - lo))) - F32(t[a])

    for a in range(3):
        for v in limit_values(*box[a]):
            x = solve_translated(v, t[a])
            assert x is not None, (a, v, t[a])
            for _ in range(3):
                r = [inside(0), inside(1), inside(2), F32(rng.uniform(0, 255))]
                r[a] = x
                if intensity_window is not None:
                    r[3] = F32(rng.uniform(*intensity_window))
                rows.append(r)
    if intensity_window is not None:
        for v in limit_values(*intensity_window):
            for _ in range(3):
                rows.append([inside(0), inside(1), inside(2), v])
    out = np.array(rows, F32)
    rnd = _filler(rng, n_random, -1.0, 1.0)
    for a in range(3):
        half = 0.6 * (box[a][1] - box[a][0])
        rnd[:, a] = (centre[a] + half * rnd[:, a] - float(F32(t[a]))).astype(F32)
    if intensity_window is not None:
        rnd[:, 3] = rng.uniform(intensity_window[0] - 20, intensity_window[1] + 20, size=n_random).astype(F32)
    out = np.concatenate([out, rnd])
    return out[rng.permutation(len(out))]


def signed_zero_subnormal_cloud(seed: int, n_random: int = 500) -> np.ndarray:
    """-0.0 and +0.0 coordinates and subnormal coordinates / intensities of both signs, for a sensor whose transform is the
    identity with translation -0.0 (so -0.0 stays -0.0 and a subnormal stays subnormal through the unfused transform)."""
    rng = np.random.default_rng(seed)
    tiny = np.array([1e-45, 1e-40, 1.1754942e-38], F32)   # smallest, mid and largest subnormal
    special = np.concatenate([tiny, -tiny, np.array([0.0, -0.0], F32)])
    rows = []
    # the other coordinates of a special row are negative: 0 * (negative) is -0.0, so a -0.0 coordinate keeps its sign
    # through the unfused transform (with a positive one, -0.0 + 0.0 would round to +0.0)
    for a in range(3):
        for v in special:
            for _ in range(2):
                r = rng.uniform(-0.5, -0.01, size=4).astype(F32)
                r[3] = F32(rng.uniform(0, 255))
                r[a] = v
                rows.append(r)
    for v in special:
        r = rng.uniform(-0.5, -0.01, size=4).astype(F32)
        r[0] = F32(0.25)
        r[3] = v
        rows.append(r)
    allneg = np.array([[-0.0, -0.0, -0.0, -0.0], [-1e-40, -1e-40, -1e-40, -1e-40], [1e-40, 1e-40, 1e-40, 1e-40]], F32)
    out = np.concatenate([np.array(rows, F32), allneg, _filler(rng, n_random, -0.5, 0.5)])
    return out[rng.permutation(len(out))]


def identity_extrinsic(t) -> np.ndarray:
    m = np.zeros((3, 4), F32)
    m[0, 0] = m[1, 1] = m[2, 2] = 1.0
    m[:, 3] = np.asarray(t, F32)
    return m


def rotated_extrinsic(yaw: float, t, pitch: float = 0.0) -> np.ndarray:
    cy, sy, cp, sp = np.cos(yaw), np.sin(yaw), np.cos(pitch), np.sin(pitch)
    r = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]]) @ np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]])
    m = np.zeros((3, 4), F32)
    m[:, :3] = r.astype(F32)
    m[:, 3] = np.asarray(t, F32)
    return m


def limits_from_data(transformed: np.ndarray, q=(0.2, 0.8)):
    """Crop limits that are transformed coordinates which actually occur: (axis, lo, hi) per axis from quantiles."""
    out = []
    for a in range(3):
        s = np.sort(transformed[:, a])
        out.append((a, float(s[int(q[0] * (len(s) - 1))]), float(s[int(q[1] * (len(s) - 1))])))
    return out


# ---- C: large offsets ----------------------------------------------------------------------------------------------------
MAP_CENTRE = (3000.0, -4500.0, 40.0)


def offset_cloud(seed: int, leaf, n: int = 60000, centre=MAP_CENTRE, extent=(60.0, 60.0, 6.0)) -> np.ndarray:
    """A map-frame cloud around `centre` (kilometres from the origin), half of it family-A lattice points there."""
    rng = np.random.default_rng(seed)
    fill = np.empty((n // 2, 4), F32)
    for a in range(3):
        fill[:, a] = (centre[a] + rng.uniform(-extent[a] / 2, extent[a] / 2, size=n // 2)).astype(F32)
    fill[:, 3] = rng.uniform(0, 255, size=n // 2).astype(F32)
    lat = lattice_cloud(seed + 1, leaf, n_lattice=n - n // 2, n_filler=0, k_span=int(min(extent) / 2 / leaf), centre=centre)
    out = np.concatenate([fill, lat])
    return out[rng.permutation(len(out))]


# ---- D: grid-size boundaries ---------------------------------------------------------------------------------------------
def grid_cloud(seed: int, div, n_filler: int = 20000, origin=(0.0, 0.0, 0.0), leaf: float = 1.0, inset: float = 0.5) -> np.ndarray:
    """Points whose data grid is exactly div cells (leaf a power of two: every extent is exact): the eight corners of the box
    [origin + inset*leaf, origin + (div - inset)*leaf], plus filler -- a dense clump near the origin and points spread over
    the whole box. With inset 0.9 PCL's d = trunc((max - min) * inv) + 1 is one less than div on every axis."""
    rng = np.random.default_rng(seed)
    o = np.asarray(origin, np.float64)
    lo = o + inset * leaf
    hi = o + (np.asarray(div, np.float64) - inset) * leaf
    corners = np.array([[(hi if (c >> a) & 1 else lo)[a] for a in range(3)] for c in range(8)])
    spread = rng.uniform(lo, hi, size=(n_filler // 2, 3))
    clump = lo + rng.uniform(0, 12 * leaf, size=(n_filler - n_filler // 2, 3))
    xyz = np.concatenate([corners, spread, clump])
    out = np.empty((len(xyz), 4), F32)
    out[:, :3] = xyz.astype(F32)
    out[:, 3] = rng.uniform(0, 255, size=len(xyz)).astype(F32)
    return out[rng.permutation(len(out))]


# div of the cell-count boundaries: index bits 31 / 32 (2^31 cells and just above) and 32 / 33 (2^32 and just above)
DIV_2P31 = (2048, 1024, 1024)
DIV_2P31_PLUS = (2048, 1024, 1025)
DIV_2P32 = (2048, 2048, 1024)
DIV_2P32_PLUS = (2048, 2048, 1025)
# PCL's INT32 guard: d = 1290 per axis passes, 1291 trips it
DIV_GUARD_BELOW = (1290, 1290, 1290)
DIV_GUARD_ABOVE = (1291, 1291, 1291)
# the largest float32 cell origin below 2^30 (float32 spacing there is 64) and 2^30 itself
ORIGIN_OK = 1073741760.0
ORIGIN_BEYOND = 1073741824.0


def bits_for(cells: int) -> int:
    return 0 if cells <= 1 else int(cells - 1).bit_length()
