"""Seeded edge-case inputs for the voxel and crop kernels (tests only).

Random clouds almost never put a coordinate where the float32 formulas are fragile. These generators do so on purpose:

  A  lattice points: coordinates on and a few ulps around the voxel planes k * leaf, where floor(f32(x * inv)) decides the
     cell and a kernel that divided, fused or rounded the product differently would pick the neighbour cell;
  B  crop-limit points: transformed coordinates exactly on a PassThrough / box limit and one ulp either side, -0.0 against
     a limit of 0.0, subnormal coordinates and intensities;
  C  large offsets: map-frame clouds kilometres from the origin (coarsest float32 cells and centroid sums);
  D  grid-size boundaries: clouds whose extent puts the cell count, the key width or PCL's INT32 guard exactly on or one
     cell past a threshold.
  N  radius outlier removal: neighbour pairs across computed cell planes up to the 2^14-cell bound, the cell table's gaps
     and bounds, every key width and pass count, the count's early exit, and grids the plan must refuse.

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


# ---- giant-cloud mode: key widths, histogram-bin boundaries, degenerate clouds --------------------------------------------
# data grids (leaf 1.0) whose voxel index space is exactly 2^bits cells: 8, 16, 24, 40, 48 and 56 are the widths where one
# more key bit needs one more radix pass, 32 the last one of a 4-byte key
KEY_WIDTH_DIVS = {8: (16, 16, 1), 16: (256, 256, 1), 24: (256, 256, 256), 31: DIV_2P31, 32: DIV_2P32, 33: DIV_2P32_PLUS,
                  40: (1 << 20, 1 << 10, 1 << 10), 48: (1 << 16, 1 << 16, 1 << 16), 56: (1 << 21, 1 << 21, 1 << 14),
                  63: (1 << 21, 1 << 21, 1 << 21)}
# data grids whose 16384-bin key histogram has a bin width of 1, a power of two (64), an odd non-power of two (63) and one
# of at least 2^40 (2^40 + 2^28)
BIN_WIDTH_DIVS = {"w1": (32, 32, 16), "w64": (128, 128, 64), "w63": (101, 101, 101), "w2p40": (1 << 21, 1 << 21, 4097)}
HIST_BINS = 1 << 14


def key_cell_cloud(div, keys, leaf: float = 1.0) -> np.ndarray:
    """One point at the centre (i + 0.5) * leaf of every given voxel index of the grid div (origin 0; exact in float32 for
    cells below 2^22 on an axis)."""
    k = np.asarray(keys, np.int64)
    d0, d1 = int(div[0]), int(div[1])
    ijk = np.stack([k % d0, (k // d0) % d1, k // (d0 * d1)], axis=1)
    out = np.zeros((len(k), 4), F32)
    out[:, :3] = ((ijk.astype(np.float64) + 0.5) * leaf).astype(F32)
    out[:, 3] = (k % 251).astype(F32)
    return out


def grid_corner_keys(div) -> list:
    d0, d1, d2 = (int(v) for v in div)
    return [i + j * d0 + k * d0 * d1 for k in (0, d2 - 1) for j in (0, d1 - 1) for i in (0, d0 - 1)]


def key_width_cloud(seed: int, div, n_filler: int = 20000) -> np.ndarray:
    """grid_cloud at leaf 1.0 with every filler point inside the box, so that the data grid is div even where an axis has
    fewer cells than the clump near the origin spans."""
    x = grid_cloud(seed, div, n_filler=n_filler)
    hi = (np.asarray(div, np.float64) - 0.5).astype(F32)
    x[:, :3] = np.minimum(x[:, :3], hi)
    return x


def bin_boundary_keys(div, bins: int = HIST_BINS, ks=None) -> list:
    """Voxel indices k*width - 1, k*width and k*width + 1 around three bin boundaries (a quarter, half and three quarters of
    the bins) of the grid's key histogram."""
    cells = int(div[0]) * int(div[1]) * int(div[2])
    width = max(1, -(-cells // bins))
    ks = ks or (bins // 4, bins // 2, 3 * bins // 4)
    return [k * width + e for k in ks for e in (-1, 0, 1)]


def bin_boundary_cloud(div, bins: int = HIST_BINS) -> np.ndarray:
    """The eight grid corners (they fix the box, so min_b = 0 and div_b = div) and one point at each bin-boundary key. With
    17 points in all, every running sum from 1 to 15 is a balancing target of 16 ranks: moving any single key into the
    neighbouring bin moves a splitter."""
    return key_cell_cloud(div, grid_corner_keys(div) + bin_boundary_keys(div, bins))


def with_nonfinite(x, every: int = 500, seed: int = 0) -> np.ndarray:
    """x with non-finite rows inserted: a copy of a row with NaN on one axis after every `every` rows (at least one), plus
    three rows with +-inf. The finite rows, and so the grid and the voxels, stay those of x."""
    rng = np.random.default_rng(seed)
    x = np.asarray(x, F32)
    n_nan = max(1, len(x) // every)
    src = rng.integers(0, max(len(x), 1), size=n_nan + 3) if len(x) else np.zeros(n_nan + 3, np.int64)
    bad = x[src].copy() if len(x) else np.zeros((n_nan + 3, 4), F32)
    axis = np.arange(n_nan + 3) % 3
    bad[np.arange(n_nan), axis[:n_nan]] = np.nan
    bad[n_nan:, :3][np.arange(3), axis[n_nan:]] = np.array([np.inf, -np.inf, np.inf], F32)
    pos = np.concatenate([np.minimum(np.arange(1, n_nan + 1) * every, len(x)), rng.integers(0, len(x) + 1, size=3)])
    return np.insert(x, pos, bad, axis=0)


def degenerate_cloud(kind: str, seed: int = 0) -> np.ndarray:
    """empty; all non-finite; one point; every point in one voxel; 3 finite points (fewer than most rank counts) among
    non-finite rows; one hot voxel holding 90 % of the points (several balancing targets in one histogram bin)."""
    rng = np.random.default_rng(seed)
    if kind == "empty":
        return np.zeros((0, 4), F32)
    if kind == "all-nonfinite":
        x = _filler(rng, 2000, -5.0, 5.0)
        x[:, 0] = np.nan
        x[::7, 1] = np.inf
        x[::11, 2] = -np.inf
        return x
    if kind == "one-point":
        return np.array([[1.25, -3.5, 0.75, 7.0]], F32)
    if kind == "one-voxel":   # cell 4 of a 0.5 leaf on every axis
        return _filler(rng, 5000, 2.0625, 2.4375)
    if kind == "three-finite":
        x = np.full((300, 4), np.nan, F32)
        x[[17, 150, 299]] = [[0.5, 0.5, 0.5, 1.0], [-3.5, 7.25, 2.5, 2.0], [9.5, -1.5, -4.5, 3.0]]
        return x
    if kind == "hot-voxel":
        hot = _filler(rng, 27000, 10.125, 10.875)
        rest = _filler(rng, 3000, -20.0, 20.0)
        x = np.concatenate([hot, rest])
        return x[rng.permutation(len(x))]
    raise ValueError(kind)


DEGENERATE_KINDS = ("empty", "all-nonfinite", "one-point", "one-voxel", "three-finite", "hot-voxel")


def giant_case(name: str):
    """(cloud, leaf) of a named giant-cloud edge case (see GIANT_CASES); a "+nf" suffix adds non-finite rows."""
    if name.endswith("+nf"):
        x, leaf = giant_case(name[:-3])
        return with_nonfinite(x, seed=len(name)), leaf
    kind, arg = name.split(":")
    if kind == "bits":
        return key_width_cloud(800 + int(arg), KEY_WIDTH_DIVS[int(arg)]), 1.0
    if kind == "bin":
        return bin_boundary_cloud(BIN_WIDTH_DIVS[arg]), 1.0
    if kind == "A":
        return lattice_cloud(820, float(arg), n_lattice=30000, n_filler=20000), float(arg)
    if kind == "C":
        return offset_cloud(821, float(arg), n=60000), float(arg)
    if kind == "Z":
        return signed_zero_subnormal_cloud(822, n_random=3000), float(arg)
    if kind == "origin":   # ok+ / ok- / beyond+ / beyond-
        o = {"ok+": ORIGIN_OK, "ok-": -ORIGIN_OK, "beyond+": ORIGIN_BEYOND, "beyond-": -ORIGIN_BEYOND}[arg]
        return grid_cloud(823, (4, 5, 6), n_filler=5000, origin=(o, 0.0, 0.0)), 1.0
    if kind == "axis":     # 2^21 cells on x (accepted) and one more (the key range)
        return grid_cloud(824, ((1 << 21) + (arg == "2p21+"), 3, 2), n_filler=5000), 1.0
    if kind == "deg":
        return degenerate_cloud(arg, 825), 0.5
    raise ValueError(name)


GIANT_CASES = (["bits:%d" % b for b in KEY_WIDTH_DIVS] + ["bin:%s" % w for w in BIN_WIDTH_DIVS] +
               ["A:0.1", "A:0.035", "C:0.05", "Z:0.05", "origin:ok+", "origin:ok-", "axis:2p21"] +
               ["deg:%s" % k for k in DEGENERATE_KINDS])
GIANT_RANGE_CASES = ("origin:beyond+", "origin:beyond-", "axis:2p21+")


# ---- R: run layouts for the centroid pass --------------------------------------------------------------------------------
# k_voxel_centroid (cloud_merger_b200/csrc/cm_voxel.cu) decides most things by where a run of equal keys sits relative to
# its own fixed structures: threads of CE_IPT items, warps, tiles of CE_TILE items, the inline walk of CE_TAIL_INLINE points
# past a tile and the rounds of CE_TAIL_ITEMS items of finish_tail_run. Its constants are mirrored here so that the layouts
# can aim at them; test_edge_inputs.py reads them out of the source, so a retune fails there instead of missing the edges.
VX_THREADS = 256
CE_IPT = 8
CE_TILE = VX_THREADS * CE_IPT            # sorted items per centroid tile
CE_TAIL_INLINE = 24                      # points past its tile a run is summed by one thread before it is handed over
CE_TAIL_U = 4
CE_TAIL_ITEMS = CE_TAIL_U * VX_THREADS   # sorted items per round of finish_tail_run
CE_SEG_SMEM_FRAMES = 256                 # frame-segmented runs: frame starts staged in shared memory up to this many frames
CE_MIN_CTAS = 3                          # resident centroid CTAs per SM (the persistent grid is 148 * CE_MIN_CTAS)
B200_SMS = 148
RUN_ROW = 1024                           # cells per row of a run-layout cloud: run r sits in cell (r % RUN_ROW, r // RUN_ROW, 0)

R_BOUND_OFFSETS = (-9, -8, -7, -1, 0, 1, 7, 8, 9)
# how far a run continues past the end of the tile its head is in: the inline walk (up to 24), the hand-over at the 25th
# point, and long runs ...
LEAVE_PAST = (0, 1, 2, 23, 24, 25, 26, 1023, 1024, 1025, 2047, 2048, 2049, 3071, 3072, 3073)
# ... among them those whose tail rounds (they start after the 24 inline points) end one short of, on and one past a round
LEAVE_ROUND = tuple(CE_TAIL_INLINE + k * CE_TAIL_ITEMS + d for k in (1, 2, 3) for d in (-1, 0, 1))
LEAVE_BACK = (1, 7, 8, 9, 255, 256, 257, 1000, 2047, 2048)   # the head of such a run: this many items before its tile's end
MINPTS_M = (2, 3, 24, 25, 26, 1025)


class RunList:
    """Run lengths in sorted order, appended at the current sorted position `pos`; `marks` names the positions a layout
    aims at (run starts) so that the CPU test can check them against the oracle's own runs."""

    def __init__(self, seed: int):
        self.rng = np.random.default_rng(seed)
        self.runs, self.pos, self.marks = [], 0, {}

    def run(self, n: int, mark: str = None):
        assert n > 0, n
        if mark:
            self.marks.setdefault(mark, []).append((self.pos, self.pos + int(n)))
        self.runs.append(int(n))
        self.pos += int(n)
        return self

    def fill(self, to: int, lo: int = 1, hi: int = 9):
        """Runs of lo..hi points up to sorted position `to`; the last one ends exactly there."""
        assert to >= self.pos, (to, self.pos)
        while self.pos < to:
            self.run(min(int(self.rng.integers(lo, hi + 1)), to - self.pos))
        return self

    def to_tile_edge(self):
        return self.fill(-(-self.pos // CE_TILE) * CE_TILE)


def next_edge(pos: int, step: int, skip: int = 0) -> int:
    """The first multiple of `step` above pos that is not a multiple of `skip`."""
    e = (pos // step + 1) * step
    while skip and e % skip == 0:
        e += step
    return e


def bounds_block(rl: RunList, tiles=(0, 1, 3, 6)):
    """R-bounds: runs of 1 to 9 points ending at every offset of R_BOUND_OFFSETS around a thread edge, a warp edge and the tile
    edge of each of the given tiles (counted from the next tile edge)."""
    t0 = -(-rl.pos // CE_TILE)
    for t in tiles:
        b = (t0 + t) * CE_TILE
        for e in (b + 5 * CE_IPT, b + 3 * VX_THREADS, b + CE_TILE):
            rl.fill(e + R_BOUND_OFFSETS[0])
            rl.marks.setdefault("bounds", []).append(e)
            for d in R_BOUND_OFFSETS[1:]:
                rl.run(e + d - rl.pos)
    return rl


def leave_block(rl: RunList):
    """R-leave: for every distance of LEAVE_PAST + LEAVE_ROUND a run whose head lies LEAVE_BACK items before the end of its
    tile and which continues that far past it; then runs from a tile's first item over exactly 1, 2 and 3 whole tiles."""
    for n, past in enumerate(LEAVE_PAST + LEAVE_ROUND):
        back = LEAVE_BACK[n % len(LEAVE_BACK)]
        end = next_edge(rl.pos, CE_TILE)
        if end - back < rl.pos:
            end += CE_TILE
        rl.fill(end - back).run(back + past, "leave")
        rl.fill(rl.pos + 1 + n % 13)
    for k in (1, 2, 3):
        rl.fill(next_edge(rl.pos, CE_TILE)).run(k * CE_TILE, "whole")
    return rl.fill(rl.pos + 37)


def dense_block(rl: RunList):
    """R-dense: a tile of 2048 one-point voxels; one of 2047 whose last run is handed over; tiles of exactly 256 and 257
    runs; and one of 257 runs whose last (the second voxel of thread 0) is handed over."""
    rl.to_tile_edge()
    for _ in range(CE_TILE):
        rl.run(1)
    for _ in range(CE_TILE - 1):
        rl.run(1)
    rl.run(1 + 600, "dense-last")
    rl.to_tile_edge()
    for _ in range(256):
        rl.run(8)
    for _ in range(255):
        rl.run(8)
    rl.run(4).run(4)
    for _ in range(256):
        rl.run(7)
    rl.run(256 + 600, "dense-last")
    return rl.fill(rl.pos + 50)


def layout(name: str, seed: int = 0):
    """(run lengths, marks) of a named layout: bounds, leave, dense, persist, end:<kind>, minpts:<m>:<length of the last run>."""
    rl = RunList(seed)
    if name == "bounds":
        bounds_block(rl).fill(rl.pos + 100)
    elif name == "leave":
        leave_block(rl)
    elif name == "dense":
        dense_block(rl)
    elif name == "persist":   # more than three tiles per CTA of the persistent grid
        while rl.pos < 3 << 20:
            bounds_block(rl)
            leave_block(rl)
    elif name.startswith("end:"):
        kind = name[4:]
        T = CE_TILE
        small = {"M1": [1], "M3": [3], "M7": [1, 2, 4]}
        if kind in small:
            for n in small[kind]:
                rl.run(n)
        elif kind in ("2T-1", "2T", "2T+1"):
            m_end = 2 * T + {"2T-1": -1, "2T": 0, "2T+1": 1}[kind]
            rl.fill(m_end - 12).run(12, "end")
        elif kind == "handover-round":   # handed over, and the second round starts exactly at M: the limit ends it
            rl.fill(2 * T - 5).run(5 + CE_TAIL_INLINE + CE_TAIL_ITEMS, "end")
        elif kind == "handover-partial":   # crosses into a final partial tile, handed over, ends at M
            rl.fill(3 * T - 100).run(100 + 700, "end")
        else:
            raise ValueError(name)
    elif name.startswith("minpts:"):
        _, m, last = name.split(":")
        m, last = int(m), int(last)
        for n in (m - 1, m, m + 1):
            for step, skip in ((CE_IPT, VX_THREADS), (VX_THREADS, CE_TILE), (CE_TILE, 0)):
                e = next_edge(rl.pos + n, step, skip)
                rl.fill(e - max(1, n // 2)).run(n, "straddle")
        rl.fill(rl.pos + 20).run(last, "end")
    else:
        raise ValueError(name)
    return rl.runs, rl.marks


R_LAYOUTS = ("bounds", "leave", "dense", "end:M1", "end:M3", "end:M7", "end:2T-1", "end:2T", "end:2T+1",
             "end:handover-round", "end:handover-partial")
R_MINPTS = tuple("minpts:%d:%d" % (m, last) for m in MINPTS_M for last in (m - 1, m, m + 1))


def _intensities(rng, n):
    return (rng.uniform(0.0, 255.0, size=n) * 2.0 ** rng.integers(-12, 1, size=n)).astype(F32)


def _make_order_sensitive(x, keys, rng):
    """Redraws the intensities of every run of 3 or more points whose float32 sequential sum in ascending row order equals
    the reversed sum in all four components (a few per cent of the short runs), until there is none."""
    order = np.argsort(keys, kind="stable")
    order = order[keys[order] >= 0]
    k = keys[order]
    starts = np.nonzero(np.r_[True, k[1:] != k[:-1]])[0] if len(k) else np.zeros(0, np.int64)
    lens = np.diff(np.r_[starts, len(k)])
    todo = np.nonzero(lens >= 3)[0]
    for _ in range(100):
        bad = []
        for n in np.unique(lens[todo]):
            rs = todo[lens[todo] == n]
            p = x[order[starts[rs][:, None] + np.arange(n)]]
            fwd = np.zeros((len(rs), 4), F32)
            rev = np.zeros((len(rs), 4), F32)
            for j in range(n):
                fwd += p[:, j]
                rev += p[:, n - 1 - j]
            bad.append(rs[(fwd.view(np.uint32) == rev.view(np.uint32)).all(axis=1)])
        todo = np.concatenate(bad) if bad else todo[:0]
        if not len(todo):
            return
        rows = order[np.concatenate([np.arange(starts[r], starts[r] + lens[r]) for r in todo])]
        x[rows, 3] = _intensities(rng, len(rows))
    raise AssertionError("runs whose sum does not depend on the order")


def run_layout_cloud(runs, seed: int, n_nonfinite: int = 0, far: bool = False, shift=(0, 0, 0)) -> np.ndarray:
    """Family R: a cloud (leaf 1.0) whose VoxelGrid has exactly the given runs in sorted order -- run r is cell r of rows of
    RUN_ROW cells (origin 0). Every point is jittered inside its cell, at least 0.1 from its planes; the coordinates of a run
    differ in their fraction bits (z and intensity in their exponents too), so its float32 sum depends on every point, and
    from 3 points on on their order (intensities are drawn again where it would not). The rows are permuted: the gather is
    scattered, and the ascending-index order inside a run is not the order of generation. n_nonfinite: rows with a NaN or an
    infinity (they sort last, into the sentinel frame); far: a point in the far corner cell of the grid DIV_2P32_PLUS (the
    keys need 33 index bits; one more run at the end); shift: whole cells added to every coordinate (another grid origin)."""
    rng = np.random.default_rng(seed)
    runs = np.asarray(runs, np.int64)
    keys = np.repeat(np.arange(len(runs), dtype=np.int64), runs)
    out = key_cell_cloud((RUN_ROW, 1 << 21, 1), keys)
    out[:, :3] = (np.floor(out[:, :3]).astype(np.float64) + rng.uniform(0.1, 0.9, size=(len(keys), 3))
                  + np.asarray(shift, np.float64)).astype(F32)
    out[:, 3] = _intensities(rng, len(keys))
    if far:
        out = np.concatenate([out, key_cell_cloud(DIV_2P32_PLUS, grid_corner_keys(DIV_2P32_PLUS)[-1:])])
        keys = np.r_[keys, len(runs)]
    if n_nonfinite:
        bad = out[rng.integers(0, len(out), size=n_nonfinite)].copy()
        bad[np.arange(n_nonfinite), np.arange(n_nonfinite) % 3] = np.array([np.nan, np.inf, -np.inf], F32)[np.arange(n_nonfinite) % 3]
        out = np.concatenate([out, bad])
        keys = np.r_[keys, np.full(n_nonfinite, -1, np.int64)]
    perm = rng.permutation(len(out))
    out, keys = out[perm], keys[perm]
    _make_order_sensitive(out, keys, rng)
    return out


def split_runs(runs, cuts):
    """The runs of each frame when the sorted sequence is cut at the given positions (a run that a cut passes through goes on,
    as a run of its own, in the next frame; equal cuts make empty frames)."""
    ends = np.cumsum(runs)
    starts = ends - np.asarray(runs)
    frames, lo = [], 0
    for hi in list(cuts) + [int(ends[-1]) if len(ends) else 0]:
        f = []
        for s, e in zip(starts, ends):
            a, b = max(int(s), lo), min(int(e), hi)
            if a < b:
                f.append(b - a)
        frames.append(f)
        lo = hi
    return frames


def centroid_walk(starts, m_items: int, frame_starts=(0,)):
    """How k_voxel_centroid meets each run [starts[r], starts[r+1]) of a sorted array of m_items items: the tile of its head,
    how far it continues past that tile, whether it is handed over to the CTA and how many items its tail rounds cover, and
    whether its tile straddles frames (frame_starts: the first position of every frame)."""
    starts = np.asarray(starts, np.int64)
    ends = np.append(starts[1:], m_items)
    tile = starts // CE_TILE
    tile_end = np.minimum((tile + 1) * CE_TILE, m_items)
    past = np.maximum(ends - tile_end, 0)
    fs = np.asarray(frame_starts, np.int64)
    first_frame = np.searchsorted(fs, tile * CE_TILE, side="right") - 1
    last_frame = np.searchsorted(fs, tile_end - 1, side="right") - 1
    return dict(start=starts, end=ends, tile=tile, past=past, handed=past > CE_TAIL_INLINE,
                tail_items=np.maximum(past - CE_TAIL_INLINE, 0), straddles=first_frame != last_frame)


def batch_layout(name: str, seed: int = 0):
    """(runs, cuts, marks) of a frame-split run layout (split_runs gives each frame's runs).
    seg3: frame 0 is one run from item 0 to 10 past the first tile, frame 1 one run from there to 500 past the third tile
    (handed over; its tile straddles frames 0 and 1), frame 2 starts with a run -- the same voxel index 0 as the end of
    frames 0 and 1, so only the frame tells the runs apart, inside the inline walk and inside a tail round -- and goes on
    with the R-bounds and R-leave blocks (tail runs in tiles of one frame).
    seg300: the R-bounds and R-leave blocks cut into 300 frames: at every R-bounds offset, around single-run frames that end
    inside an inline walk or a tail round, with empty frames, and at further random positions among the R-bounds runs."""
    T = CE_TILE
    if name == "seg3":
        rl = RunList(seed)
        rl.run(T + 10).run(2 * T + 490, "tail-straddle").run(30)
        bounds_block(rl)
        leave_block(rl)
        return rl.runs, [T + 10, 3 * T + 500], rl.marks
    if name == "seg300":
        rl = RunList(seed)
        bounds_block(rl)
        split = rl.pos
        leave_block(rl)
        cuts = [e + d for e in rl.marks["bounds"] for d in R_BOUND_OFFSETS]
        leave = rl.marks["leave"]
        for k, past in ((7, 10), (10, 300), (16, 700)):   # single-run frames ending inline / in a tail round
            s, e = leave[k]
            t_end = (s // T + 1) * T
            assert e - t_end > past
            cuts += [s + 1, t_end + past]
        cuts += [cuts[0]] * 2 + [cuts[50]] + [split] * 2   # empty frames
        rng = np.random.default_rng(seed + 1)
        while len(cuts) < 299:
            cuts.append(int(rng.integers(1, split)))
        return rl.runs, sorted(cuts), rl.marks
    raise ValueError(name)


def run_layout_frames(runs, cuts, seed: int, n_nonfinite: int = 0, shift=(0, 0, 0)) -> list:
    """One run-layout cloud per frame of split_runs(runs, cuts); frame f is shifted by f * shift cells, and frames with points
    get n_nonfinite non-finite rows each."""
    out = []
    for f, fr in enumerate(split_runs(runs, cuts)):
        if not fr:
            out.append(np.zeros((0, 4), F32))
            continue
        out.append(run_layout_cloud(fr, seed + f, n_nonfinite=n_nonfinite, shift=tuple(f * s for s in shift)))
    return out


# ---- N: radius outlier removal (cloud_merger_b200/csrc/cm_outlier.cu) -----------------------------------------------------
# The radius outlier removal keys every point on a grid of cells a little wider than the radius, sorts the keys and lets
# every point count inside the 3 x 3 rows of cells around its own, through a direct-address table of the cells' first
# sorted positions (k_ror_table) or binary searches. ror_plan restates that plan in numpy: the cell, the grid of every
# cloud (k_grid_setup), the keys and the sort plan, the table, and the nine rows each point searches with the table
# entries they read. Its constants mirror the source; test_edge_inputs.py reads them out of it.
ROR_MARGIN = 1.00390625                  # cell = f32(f32(radius) * (1 + 2^-8))
ROR_BOUND = 1 << 14                      # |cell index| the margin covers; k_ror_count refuses from here on
ROR_TABLE_LOG2 = 25                      # the table is used while n_clouds << idx_bits <= 2^25
ROR_THREADS = 256                        # CTA of k_ror_table
ROR_LONG_GAP = 2048                      # k_ror_table: a gap with to - from >= this goes to the CTA's shared list ...
ROR_LIST = 32                            # ... of this many entries; more fall back to the warp that found them
ROR_ROW_DZ, ROR_ROW_DY = 0x28215, 0x22161   # (dz + 1, dy + 1) of row rr in bits 2rr, 2rr + 1
GRID_RANGE_CELLS = 1 << 21               # k_grid_setup: more cells on an axis, or a coordinate beyond 2^30 cells, is
GRID_RANGE_ORIGIN = 1 << 30              # out of range and the frame is keyed as one cell (zero_keys)
ROR_RADII = (float(F32(0.15)), 0.15, 1e-3, 0.5, 3.0)   # 0.15 as the float the reference holds, and as a double
# a radius whose float32 cell is below it (f32(0.45) < 0.45): there the computed planes 2^k and 2^k + 1 (k = 1, 5, 9, 13)
# are closer than the radius, so that without the margin two neighbours can sit two cells apart
ROR_RADIUS_TIGHT = 0.45


def ror_rows():
    """(dz, dy) of the nine rows in the order k_ror_count visits them."""
    return [(((ROR_ROW_DZ >> (2 * rr)) & 3) - 1, ((ROR_ROW_DY >> (2 * rr)) & 3) - 1) for rr in range(9)]


def ror_cell(radius, margin: bool = True) -> np.float32:
    r = F32(radius)
    return F32(r * F32(ROR_MARGIN)) if margin else r


def ror_r2(radius) -> np.float32:
    return F32(float(radius) * float(radius))


def ror_cells(x, cell) -> np.ndarray:
    """floor(f32(x * (1 / cell))) per coordinate, as int64 (the cell of every point before min_b is taken off)."""
    inv = F32(F32(1.0) / F32(cell))
    with np.errstate(invalid="ignore", over="ignore"):
        return np.floor((np.asarray(x, F32)[:, :3] * inv).astype(F32)).astype(np.float64)


def _bits(cells: int) -> int:
    return 0 if cells <= 1 else int(cells - 1).bit_length()


def ror_grid(x, cell) -> dict:
    """k_grid_setup of one cloud on the cell grid: min_b, max_b, div_b (kept at the real width even when out of range, as
    the kernel leaves it), whether the grid is out of range (zero_keys: every key 0) and its index bits."""
    x = np.asarray(x, F32)
    fin = np.isfinite(x[:, :3]).all(axis=1)
    if not fin.any():
        return dict(empty=True, min_b=np.zeros(3, np.int64), max_b=np.zeros(3, np.int64), div=np.zeros(3, np.int64),
                    zero_keys=False, bits=0)
    fc = ror_cells(x[fin], cell)
    fmn, fmx = fc.min(axis=0), fc.max(axis=0)
    err = bool((np.abs(fmn) >= GRID_RANGE_ORIGIN).any() or (np.abs(fmx) >= GRID_RANGE_ORIGIN).any())
    lim = float(2 ** 31 - 1)
    mn = np.clip(fmn, -lim - 1, lim).astype(np.int64)      # (int) of the float saturates on the device
    mx = np.clip(fmx, -lim - 1, lim).astype(np.int64)
    div = mx - mn + 1
    err = err or bool((div > GRID_RANGE_CELLS).any())
    cells = 1 if err else int(div[0]) * int(div[1]) * int(div[2])
    return dict(empty=False, min_b=mn, max_b=mx, div=div, zero_keys=err, bits=_bits(cells))


def ror_plan(clouds, radius, table: bool = True, fixed: bool = True, margin: bool = True) -> dict:
    """The whole plan of one radius_outlier_multi call (a single cloud is a list of one).
    fixed=False restates the library before the host refused out-of-range grids: such a frame is then counted with key 0
    and its real div_b. Returns the grids, the sort plan (idx_bits, key bytes, passes, table keys), whether the call is
    refused (plan_error: before the table; bound_error: by the count kernel), and per point of every cloud its cells, key,
    the nine row segments [k_lo, k_hi] it searches (-1 where a clamp skips the row) and the largest table entry it reads."""
    cell = ror_cell(radius, margin)
    clouds = [np.asarray(c, F32).reshape(-1, 4) for c in clouds]
    n = len(clouds)
    grids = [ror_grid(c, cell) for c in clouds]
    has_invalid = any((~np.isfinite(c[:, :3]).all(axis=1)).any() for c in clouds)
    key_frames = n + (1 if has_invalid else 0)
    frame_bits = _bits(key_frames)
    idx_bits = max([g["bits"] for g in grids if not g["empty"]] + [0])
    total = frame_bits + idx_bits
    plan_error = any(g["zero_keys"] for g in grids) or total > 64
    total = min(total, 64)
    idx_bits = total - frame_bits
    passes = max(1, -(-total // 8))
    n_points = sum(len(c) for c in clouds)
    use_table = (table and n_points > 0 and idx_bits <= ROR_TABLE_LOG2 and (n << idx_bits) <= (1 << ROR_TABLE_LOG2))
    table_keys = (n << idx_bits) if use_table else 0
    worst = max([int(max(np.abs(g["min_b"]).max(), np.abs(g["max_b"]).max())) for g in grids if not g["empty"]] + [0])
    refused = fixed and plan_error
    rows = ror_rows()
    per = []
    for f, (c, g) in enumerate(zip(clouds, grids)):
        fin = np.isfinite(c[:, :3]).all(axis=1)
        m = len(c)
        d = g["div"].astype(np.int64)
        cc = np.zeros((m, 3), np.int64)
        key = np.full(m, key_frames - 1 if has_invalid else n, np.int64) << idx_bits   # non-finite: the sentinel frame
        if fin.any() and not g["empty"]:
            if not g["zero_keys"]:
                cc[fin] = ror_cells(c[fin], cell).astype(np.int64) - g["min_b"]
            idx = cc[:, 0] + cc[:, 1] * d[0] + cc[:, 2] * d[0] * d[1]
            key[fin] = (f << idx_bits) + (0 if g["zero_keys"] else idx[fin])
        seg = np.full((m, 9, 2), -1, np.int64)
        reads = np.full(m, -1, np.int64)
        counted = fin & (not g["zero_keys"] or not fixed) & (not refused)
        if counted.any():
            c0, c1, c2 = cc[:, 0], cc[:, 1], cc[:, 2]
            x_lo, x_hi = np.maximum(c0 - 1, 0), np.minimum(c0 + 1, d[0] - 1)
            for rr, (dz, dy) in enumerate(rows):
                ok = counted.copy()
                if dz < 0: ok &= c2 > 0
                if dz > 0: ok &= c2 + 1 < d[2]
                if dy < 0: ok &= c1 > 0
                if dy > 0: ok &= c1 + 1 < d[1]
                row = ((c2 + dz) * d[1] + (c1 + dy)) * d[0]
                seg[ok, rr, 0] = (f << idx_bits) + row[ok] + x_lo[ok]
                seg[ok, rr, 1] = (f << idx_bits) + row[ok] + x_hi[ok]
            hi = np.where(seg[:, :, 1] >= 0, seg[:, :, 1] + 1, -1).max(axis=1)
            reads = np.where(counted, hi, -1)
        per.append(dict(cells=cc, key=key, fin=fin, seg=seg, max_read=reads))
    return dict(cell=cell, grids=grids, idx_bits=idx_bits, frame_bits=frame_bits, total_bits=total, passes=passes,
                key_bytes=4 if total <= 32 else 8, table=use_table, table_keys=table_keys, plan_error=plan_error,
                bound_error=worst >= ROR_BOUND, worst=worst, refused=refused, points=per)


def ror_launches(plan, clouds) -> int:
    """Kernel launches of the call as cm_launch_count reports them: a bounding box per non-empty cloud, the grid setup,
    the key kernel, the radix passes, the table when it is used, the count."""
    return sum(1 for c in clouds if len(c)) + 3 + plan["passes"] + (1 if plan["table"] else 0)


def ror_pairs(x, radius) -> np.ndarray:
    """(i, j), i < j, of the finite points of one cloud strictly inside the radius in the count's float order."""
    from scipy.spatial import cKDTree
    x = np.asarray(x, F32)
    fin = np.nonzero(np.isfinite(x[:, :3]).all(axis=1))[0]
    if len(fin) < 2:
        return np.zeros((0, 2), np.int64)
    p = cKDTree(x[fin, :3].astype(np.float64)).query_pairs(float(radius) * (1 + 1e-5) + 1e-30, output_type="ndarray")
    p = fin[p]
    d = x[p[:, 0], :3] - x[p[:, 1], :3]
    acc = ((d[:, 0] * d[:, 0]).astype(F32) + (d[:, 1] * d[:, 1]).astype(F32)).astype(F32)
    acc = (acc + (d[:, 2] * d[:, 2]).astype(F32)).astype(F32)
    return p[acc < ror_r2(radius)]


def ror_brute_count(x, radius) -> np.ndarray:
    """O(n^2) count per point (itself included) in the count's float order; 0 for non-finite points."""
    x = np.asarray(x, F32)
    fin = np.isfinite(x[:, :3]).all(axis=1)
    r2 = ror_r2(radius)
    out = np.zeros(len(x), np.int64)
    for s in range(0, len(x), 512):
        with np.errstate(invalid="ignore", over="ignore"):
            d = x[s:s + 512, None, :3] - x[None, :, :3]
            acc = ((d[..., 0] * d[..., 0]).astype(F32) + (d[..., 1] * d[..., 1]).astype(F32)).astype(F32)
            acc = (acc + (d[..., 2] * d[..., 2]).astype(F32)).astype(F32)
            inside = (acc < r2) & fin[None, :] & fin[s:s + 512, None]
        out[s:s + 512] = inside.sum(axis=1)
    return out


def cell_plane(p, cell) -> np.ndarray:
    """The computed plane of cell index p (scalar or array): the smallest float32 x with floor(f32(x * inv)) >= p."""
    inv = F32(F32(1.0) / F32(cell))
    p = np.asarray(p, np.float64)
    x = (p * float(cell)).astype(F32)
    for _ in range(64):
        up = np.floor((x * inv).astype(F32)) >= p
        below = np.nextafter(x, F32(-np.inf))
        down = np.floor((below * inv).astype(F32)) >= p
        if not (~up).any() and not down.any():
            return x
        x = np.where(~up, np.nextafter(x, F32(np.inf)), np.where(down, below, x)).astype(F32)
    raise AssertionError("cell plane search did not converge")


def _directions():
    out = []
    for v in np.ndindex(3, 3, 3):
        u = np.array(v, np.float64) - 1
        if u.any():
            out.append(u / np.linalg.norm(u))
    return np.array(out)   # 6 axes, 12 face diagonals, 8 space diagonals


MARGIN_PLANES = (0, 1000, 2500, 4000, 6000, 8000, 10000, 12000, 14000, ROR_BOUND - 2 - 3 * (26 * 9 - 1))


def margin_cloud(radius, sign: int = 1) -> np.ndarray:
    """N-margin: pairs at radius * (1 + k * 2^-23), k = -4..4, along the 26 axis and diagonal directions, centred on a corner
    of computed cell planes (every coordinate on a plane), one corner every third cell from the MARGIN_PLANES indices on
    (sign -1: mirrored), so that the cells of the pairs reach |index| 2^14 - 1 on every axis. Along the axes a second set
    aims at the planes of a margin-free cell (cell = radius): the first point is the last float below such a plane, the
    second the last float still inside the radius and up to 4 floats back from it -- where a grid without the margin can
    put two neighbours two cells apart."""
    cell, cell0 = ror_cell(radius), ror_cell(radius, margin=False)
    r2 = ror_r2(radius)
    dirs = _directions()
    ks = np.arange(-4, 5)
    J = len(dirs) * len(ks)
    j = np.arange(J)
    u, k = dirs[j // len(ks)], ks[j % len(ks)]
    p = sign * (np.asarray(MARGIN_PLANES)[:, None] + 3 * j[None, :]).reshape(-1)
    u, k = np.tile(u, (len(MARGIN_PLANES), 1)), np.tile(k, len(MARGIN_PLANES))
    s = float(radius) * (1 + k * 2.0 ** -23)
    c = np.column_stack([cell_plane(p, cell), cell_plane(p + 1, cell), cell_plane(-p, cell)]).astype(np.float64)
    pairs = np.stack([c - u * s[:, None] / 2, c + u * s[:, None] / 2], axis=1).reshape(-1, 3).astype(F32)
    # the aimed set: 6 axis directions x 5 steps back, at the planes 2^k (where the computed plane spacing is shortest) and
    # spread over the range; every pair at its own place on the other two axes
    Q = np.array([1 << k for k in range(1, 14)] + [m + 1 for m in MARGIN_PLANES[1:]], np.int64)
    q = sign * np.repeat(Q, 30)
    j = np.arange(len(q))
    axis, neg, k = (j // 5) % 3, (j // 15) % 2 == 1, j % 5
    keep = np.abs(q) < int((ROR_BOUND - 2) * float(cell0) / float(cell))
    q, axis, neg, k, j = q[keep], axis[keep], neg[keep], k[keep], j[keep]
    a = np.nextafter(cell_plane(q, cell0), F32(-np.inf))
    b = (a + F32(float(radius))).astype(F32)
    for _ in range(64):
        out = ((b - a) * (b - a)).astype(F32) >= r2
        if not out.any():
            break
        b = np.where(out, np.nextafter(b, F32(-np.inf)), b).astype(F32)
    for step in range(4):
        b = np.where(k > step, np.nextafter(b, F32(-np.inf)), b).astype(F32)
    base = np.column_stack([cell_plane(sign * (5 + 3 * j), cell), cell_plane(sign * (7 + 3 * j), cell),
                            cell_plane(sign * (11 + 3 * j), cell)]).astype(F32)
    q1, q2 = base.copy(), base.copy()
    rows = np.arange(len(q))
    q1[rows, axis] = np.where(neg, b, a)
    q2[rows, axis] = np.where(neg, a, b)
    aimed = np.stack([q1, q2], axis=1).reshape(-1, 3)
    out = np.concatenate([pairs, aimed])
    return np.column_stack([out, np.arange(len(out), dtype=F32)]).astype(F32)


def bound_cloud(radius, axis: int, index: int) -> np.ndarray:
    """N-bound: a small cluster near the origin plus a pair of neighbours whose cells reach `index` on one axis, so that
    the largest |cell index| of the grid is exactly |index| (2^14 - 1 passes, 2^14 is refused)."""
    cell = ror_cell(radius)
    rng = np.random.default_rng(abs(index) * 3 + axis + (index < 0))
    near = rng.uniform(-3, 3, (200, 3)) * float(cell)
    far = np.zeros((2, 3))
    lo, hi = float(cell_plane(index, cell)), float(cell_plane(index + 1, cell))
    far[:, axis] = [lo + 0.25 * (hi - lo), lo + 0.6 * (hi - lo)]
    x = np.concatenate([near, far]).astype(F32)
    assert np.abs(ror_cells(x, cell)).max() == max(abs(index), 3) or np.abs(ror_cells(x, cell)).max() == abs(index)
    return np.column_stack([x, np.arange(len(x), dtype=F32)]).astype(F32)


def range_clouds(radius=float(F32(0.15))) -> dict:
    """N-range: clouds whose cell grid k_grid_setup cannot key: more than 2^21 cells on x and y (the two-point example
    {(0,0,0), (4e5,4e5,0)}), and a cloud beyond 2^30 cells from the origin (spread over thousands of cells on x and y)."""
    cell = float(ror_cell(radius))
    wide = np.array([[0, 0, 0, 0], [4e5, 4e5, 0, 1]], F32)
    x0 = 1.01 * GRID_RANGE_ORIGIN * cell
    rng = np.random.default_rng(5)
    far = np.column_stack([x0 + 16.0 * rng.integers(0, 60, 40), rng.uniform(0, 2000, 40), np.zeros(40),
                           np.arange(40)]).astype(F32)
    return {"wide": wide, "far": far}


def gap_cloud(radius, steps, seed: int = 0) -> np.ndarray:
    """N-gap: one point per cell, at exactly the cell keys cumsum([0] + steps). The rows are as long as the last key below
    2^15 - 1 plus one (so the first row spans it and the keys come out as designed), centred on the origin. A point sits
    close to the face it shares with the next cell of its row when the key step to that cell is 1, so neighbours are in
    key-adjacent cells and a wrong table entry changes a count."""
    cell = float(ror_cell(radius))
    keys = np.concatenate([[0], np.cumsum(steps)]).astype(np.int64)
    row = int(keys[keys < (1 << 15) - 2].max()) + 1
    c0, c1 = keys % row, keys // row
    rng = np.random.default_rng(seed)
    frac = np.full(len(keys), 0.5)
    nxt = np.r_[np.diff(keys) == 1, False]
    prv = np.r_[False, np.diff(keys) == 1]
    frac[nxt & ~prv] = 0.97                 # the first of a pair: at its high face ...
    frac[prv & ~nxt] = 0.03                 # ... the second at its low face
    frac[nxt & prv] = 0.5 + rng.choice([-0.47, 0.47], size=int((nxt & prv).sum()))
    x = np.column_stack([(c0 - row // 2 + frac) * cell, (c1 + 0.5) * cell, np.full(len(keys), 0.5 * cell)]).astype(F32)
    cells = ror_cells(x, ror_cell(radius)).astype(np.int64)
    assert (cells[:, 0] == c0 - row // 2).all() and (cells[:, 1] == c1).all()
    perm = rng.permutation(len(x))
    return np.column_stack([x[perm], perm.astype(F32)]).astype(F32)


def gap_steps(kind: str) -> list:
    """Key steps of the N-gap layouts (k_ror_table: thread i fills (key[i-1], key[i]]; long means to - from >= 2048)."""
    short = lambda n, rng: list(rng.choice([1, 1, 1, 2, 3], size=n))
    rng = np.random.default_rng(len(kind))
    if kind == "edge":           # gaps of 2047, 2048, 2049, 2050 entries (to - from = 2046 .. 2049) among short ones
        s = short(300, rng)
        for j, g in enumerate((2047, 2048, 2049, 2050, 2048, 2049)):
            s[40 + 37 * j] = g
        return s
    if kind.startswith("cta"):   # L long gaps in the second CTA of 256 elements: list full, exactly full, one past
        L = int(kind[3:])
        s = short(700, rng)
        for j in range(L):
            s[300 + 6 * j] = 2049 + 17 * j
        return s
    if kind.startswith("m"):     # M % 256 in {0, 1, 255}: the gap above the largest key is thread M's
        m = int(kind[1:])
        s = short(m - 1, rng)
        s[m // 2] = 5000
        return s
    raise ValueError(kind)


GAP_KINDS = ("edge", "cta31", "cta32", "cta33", "m512", "m513", "m767")


def width_cloud(radius, bits: int, seed: int = 0, n: int = 3000) -> np.ndarray:
    """N-width: a cloud whose cell grid has exactly 2^bits cells (idx_bits = bits): its corner cells plus clusters of
    neighbours and loose points in between, centred on the origin so that no cell index reaches 2^14."""
    cell = float(ror_cell(radius))
    b = [bits // 3 + (1 if k < bits % 3 else 0) for k in range(3)]
    div = np.array([(1 << v) - (1 if v == 15 else 0) for v in b], np.int64)   # 2^15 - 1: cells -16383 .. 16383
    assert _bits(int(np.prod(div))) == bits and (div < 1 << 15).all()
    lo = -(div // 2)
    rng = np.random.default_rng(seed + bits)
    corners = np.array([[lo[k] + (div[k] - 1) * ((m >> k) & 1) for k in range(3)] for m in range(8)], np.float64)
    centres = lo + rng.random((n // 6, 3)) * (div - 1)
    pts = [corners + 0.5]
    pts += [centres + rng.normal(0, 0.4, centres.shape) for _ in range(3)]
    pts += [lo + rng.random((n // 2, 3)) * div]
    x = np.concatenate(pts)
    x = np.clip(x, lo + 0.01, lo + div - 0.01) * cell
    x = x.astype(F32)
    c = ror_cells(x, cell)
    assert (c.min(axis=0) == lo).all() and (c.max(axis=0) == lo + div - 1).all()
    return np.column_stack([x, rng.uniform(0, 255, len(x))]).astype(F32)


def count_cloud(radius, kind: str, seed: int = 0) -> np.ndarray:
    """N-count: hot: a cell of 2500 points (400 of them exact duplicates) amid loose ones -- the early exit decides in the
    middle of a row; flat1 / flat2: d = 1 on one / two axes; single: one cell; nonfinite: a hot cloud with NaN / inf rows."""
    cell = float(ror_cell(radius))
    rng = np.random.default_rng(seed)
    if kind in ("hot", "nonfinite"):
        hot = rng.uniform(0.02, 0.98, (2100, 3)) * cell + 5 * cell
        dup = np.repeat(hot[:4], 100, axis=0)
        loose = rng.uniform(0, 12 * cell, (1500, 3))
        x = np.concatenate([hot, dup, loose])
    elif kind == "flat1":
        x = np.column_stack([rng.uniform(0, 40 * cell, 3000), rng.uniform(0, 40 * cell, 3000), np.full(3000, 0.5 * cell)])
    elif kind == "flat2":
        x = np.column_stack([rng.uniform(0, 300 * cell, 3000), np.full(3000, 0.5 * cell), np.full(3000, 0.5 * cell)])
    elif kind == "single":
        x = rng.uniform(0.01, 0.99, (800, 3)) * cell + 2 * cell
    else:
        raise ValueError(kind)
    x = x.astype(F32)
    out = np.column_stack([x, rng.uniform(0, 255, len(x))]).astype(F32)
    if kind == "nonfinite":
        bad = out[rng.integers(0, len(out), 60)].copy()
        bad[np.arange(60), np.arange(60) % 3] = np.array([np.nan, np.inf, -np.inf], F32)[np.arange(60) % 3]
        out = np.concatenate([out, bad])
    return out[rng.permutation(len(out))]


COUNT_KINDS = ("hot", "flat1", "flat2", "single", "nonfinite")
COUNT_MIN_PTS = (0, 1, 2, 100, 5000, 2 ** 31 - 1)


def row_end_clouds(radius) -> list:
    """N-count, frame edges: three clouds on the same 8 x 4 x 2 cell grid, each with neighbours in the first and the last
    cell of its rows and in its first and last key cell, so that frame f's last cell and frame f + 1's first one are next
    to each other in key order (and the same place in space: counting across clouds would change the result)."""
    cell = float(ror_cell(radius))
    out = []
    for f in range(3):
        rng = np.random.default_rng(40 + f)
        pts = []
        for cy in range(4):
            for cz in range(2):
                for cx in (0, 7):
                    base = np.array([cx, cy, cz], np.float64)
                    pts.append(base + rng.uniform(0.05, 0.95, (3, 3)))
        pts.append(np.array([[0.02, 0.02, 0.02], [7.98, 3.98, 1.98]]))
        x = (np.concatenate(pts) * cell).astype(F32)
        out.append(np.column_stack([x, rng.uniform(0, 255, len(x))]).astype(F32))
    return out


def ror_cases() -> dict:
    """name -> (clouds, radius, min_pts values) of every N family the GPU runs bit-exact (N-range and the refused N-bound
    clouds are in ror_refused_cases)."""
    r15 = float(F32(0.15))
    cases = {}
    for r in ROR_RADII + (ROR_RADIUS_TIGHT,):
        for sign in (1, -1):
            cases["margin:%g%s:%+d" % (r, "f" if r == r15 else "", sign)] = ([margin_cloud(r, sign)], r, (1, 2))
    for axis in range(3):
        for sign in (1, -1):
            cases["bound:ok:%d%+d" % (axis, sign)] = ([bound_cloud(r15, axis, sign * (ROR_BOUND - 1))], r15, (1,))
    for kind in GAP_KINDS:
        cases["gap:" + kind] = ([gap_cloud(r15, gap_steps(kind))], r15, (0, 1, 2))
    for bits in (4, 12, 20, 28, 36, 44):
        cases["width:%d" % bits] = ([width_cloud(r15, bits)], r15, (1, 3))
    cases["width:25"] = ([width_cloud(r15, 25)], r15, (1,))
    cases["width:26"] = ([width_cloud(r15, 26)], r15, (1,))
    cases["width:2x24"] = ([width_cloud(r15, 24, 1), width_cloud(r15, 20, 2)], r15, (1,))
    cases["width:2x25"] = ([width_cloud(r15, 25, 1), width_cloud(r15, 12, 2)], r15, (1,))
    cases["width:3x12+36"] = ([width_cloud(r15, 12, 3), width_cloud(r15, 36, 4), width_cloud(r15, 8, 5)], r15, (2,))
    for kind in COUNT_KINDS:
        cases["count:" + kind] = ([count_cloud(r15, kind)], r15, COUNT_MIN_PTS)
    cases["count:row-ends"] = (row_end_clouds(r15), r15, (0, 1, 2, 3))
    return cases


def ror_refused_cases() -> dict:
    """name -> (clouds, radius): calls the library must refuse with CM_E_KEY_RANGE."""
    r15 = float(F32(0.15))
    rc = range_clouds(r15)
    normal = width_cloud(r15, 12, 7)
    cases = {"bound:over:%d%+d" % (a, s): ([bound_cloud(r15, a, s * ROR_BOUND)], r15) for a in range(3) for s in (1, -1)}
    cases["range:wide"] = ([rc["wide"]], r15)
    cases["range:far"] = ([rc["far"]], r15)
    cases["range:multi"] = ([normal, rc["wide"], normal[:100], rc["far"]], r15)
    return cases
