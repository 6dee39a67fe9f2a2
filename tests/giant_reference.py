"""Independent numpy reference of the giant-cloud partition plan (tests only).

Written from the definitions of cloud_merger_gpu.h (cm_giant_voxelgrid, cm_dev_key_histogram, cm_dev_route_by_key) and
DESIGN.md section 6, not from the kernels:

  grid       PCL 1.8.1 VoxelGrid::applyFilter on the box of the finite points of the WHOLE cloud: inv = f32(1 / f32(leaf)),
             min_b = floor(f32(min_p * inv)), max_b = floor(f32(max_p * inv)), div_b = max_b - min_b + 1
  key range  an error when |floor(f32(p * inv))| >= 2^30 for a bound, or when div_b > 2^21 on an axis
  keys       idx = i + j * div_x + k * div_x * div_y with ijk = floor(f32(p * inv)) - min_b, exact integers
  histogram  bins of equal key width, width = max(1, ceil(cells / bins)); a key beyond the last bin counts in the last one
  splitters  for every target total * r // W (r = 1 .. W-1): the first bin boundary at or after it, (b + 1) * width with b
             the first bin whose inclusive running sum reaches the target; an empty cloud puts every splitter at width
  grouping   the destination of a finite point is the number of splitters <= its key; a non-finite point stays on `me`;
             every part keeps the source order

All integer arithmetic is exact (int64 for keys below 2^63, Python ints for the bin width and the totals).
"""
from __future__ import annotations

import numpy as np

F32 = np.float32
BINS = 1 << 14          # the histogram of cm_giant_voxelgrid
KEY_LIMIT = 1 << 30     # |cell origin| must stay below it
AXIS_LIMIT = 1 << 21    # cells per axis


def inv_leaf(leaf) -> np.ndarray:
    return (F32(1.0) / np.broadcast_to(np.asarray(leaf, F32), (3,))).astype(F32)


def finite_rows(xyzi) -> np.ndarray:
    return np.isfinite(np.asarray(xyzi, F32)[:, :3]).all(axis=1)


def cells_of(xyz, leaf) -> np.ndarray:
    """floor(f32(p * inv)) per coordinate, as int64 (float32 product, rounded to nearest, then floor)."""
    prod = (np.asarray(xyz, F32) * inv_leaf(leaf)).astype(F32)
    return np.floor(prod.astype(np.float64)).astype(np.int64)


def bits_for(cells: int) -> int:
    return 0 if cells <= 1 else int(cells - 1).bit_length()


def grid(xyzi, leaf) -> dict:
    """The global grid of the finite points: min_p, max_p (None for a cloud without finite points), min_b, div_b, cells,
    key_bits and key_range_error. An empty grid is the one-cell grid at the origin."""
    x = np.asarray(xyzi, F32)
    fin = finite_rows(x)
    if not fin.any():
        return dict(min_p=None, max_p=None, min_b=np.zeros(3, np.int64), div_b=np.ones(3, np.int64), cells=1, key_bits=0,
                    key_range_error=False, finite=0)
    v = x[fin, :3]
    min_p, max_p = v.min(axis=0), v.max(axis=0)
    fmn, fmx = cells_of(min_p[None], leaf)[0], cells_of(max_p[None], leaf)[0]
    div = fmx - fmn + 1
    err = bool((np.abs(fmn) >= KEY_LIMIT).any() or (np.abs(fmx) >= KEY_LIMIT).any() or (div > AXIS_LIMIT).any())
    cells = int(div[0]) * int(div[1]) * int(div[2])
    return dict(min_p=min_p, max_p=max_p, min_b=fmn, div_b=div, cells=cells, key_bits=bits_for(cells), key_range_error=err,
                finite=int(fin.sum()))


def keys(xyzi, leaf, min_b, div_b) -> np.ndarray:
    """Exact voxel index of every point on the grid (min_b, div_b); -1 for a non-finite point."""
    x = np.asarray(xyzi, F32)
    fin = finite_rows(x)
    c = cells_of(np.where(fin[:, None], x[:, :3], F32(0)), leaf) - np.asarray(min_b, np.int64)
    d0, d1 = int(div_b[0]), int(div_b[1])
    k = c[:, 0] + c[:, 1] * np.int64(d0) + c[:, 2] * np.int64(d0 * d1)
    return np.where(fin, k, np.int64(-1))


def bin_width(cells: int, bins: int = BINS) -> int:
    return max(1, -(-int(cells) // int(bins)))


def histogram(key, cells: int, bins: int = BINS) -> np.ndarray:
    """Counts of the finite keys per bin of width bin_width(cells, bins) (int64 [bins])."""
    k = np.asarray(key, np.int64)
    k = k[k >= 0]
    b = np.minimum(k // np.int64(bin_width(cells, bins)), bins - 1)
    return np.bincount(b, minlength=bins).astype(np.int64)


def splitters(hist, width: int, world: int) -> list:
    """The W - 1 balancing splitters of a histogram (Python ints)."""
    hist = np.asarray(hist, np.int64)
    bins = len(hist)
    cum = np.cumsum(hist)
    total = int(cum[-1]) if bins else 0
    if total == 0:
        return [int(width)] * (world - 1)
    out = []
    for r in range(1, world):
        target = total * r // world
        b = int(np.searchsorted(cum, target, side="left"))   # first bin whose running sum reaches the target
        out.append(min(b + 1, bins) * int(width))
    return out


def destinations(key, split, me: int) -> np.ndarray:
    """Rank of every point: the number of splitters <= its key; non-finite points (key -1) stay on `me`."""
    k = np.asarray(key, np.int64)
    s = np.asarray([int(v) for v in split], dtype=np.uint64)
    d = np.searchsorted(s, np.maximum(k, 0).astype(np.uint64), side="right").astype(np.int64)
    return np.where(k >= 0, d, np.int64(me))


def grouping(dest, world: int):
    """(parts: source indices of every part in source order, send_begin: where part r starts in the grouped array)."""
    dest = np.asarray(dest, np.int64)
    parts = [np.nonzero(dest == r)[0] for r in range(world)]
    begin = [0]
    for p in parts:
        begin.append(begin[-1] + len(p))
    return parts, begin


def plan(xyzi, leaf, world: int, me: int = 0, bins: int = BINS) -> dict:
    """The whole partition plan of a cloud routed from rank `me` to `world` ranks (the dry cm_giant_voxelgrid)."""
    g = grid(xyzi, leaf)
    k = keys(xyzi, leaf, g["min_b"], g["div_b"])
    width = bin_width(g["cells"], bins)
    h = histogram(k, g["cells"], bins)
    split = splitters(h, width, world)
    dest = destinations(k, split, me)
    parts, begin = grouping(dest, world)
    n = len(k)
    return dict(g, keys=k, width=width, hist=h, splitters=split, dest=dest, parts=parts, send_begin=begin,
                total=int(h.sum()), points_sent_away=n - len(parts[me]))
