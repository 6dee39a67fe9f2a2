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
