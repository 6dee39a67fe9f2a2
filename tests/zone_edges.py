"""Edge inputs of the zone slicing (family Z): cm_zones.cu's count / scan / scatter and the box and chain membership
tests. Every filter's output is compacted here, so these edges matter to all of them.

The constants mirror the sources (tests/test_zone_edges.py pins them):
  - ZN_TILE points per k_zone_count / k_zone_scatter tile, in warp rows of WARP_ROW points;
  - SCAN_TILES tiles per round of k_zone_scan's loop (carry in s_run): a cloud of more than SCAN_TILES * ZN_TILE points
    runs a second round;
  - MAX_ZONES zones per split (mask bit z = zone z).

Cases: Z-tile (membership flips on warp-row and tile edges, points in 0, 1, several and all zones, zone 15 alone),
Z-scan (16 zones with points in every scan round), Z-path (the same windows as boxes and, forced by NOOP, as chains),
Z-grow (16 keep-all zones: the outputs regrow in cm_get_zone_out)."""
from __future__ import annotations

import numpy as np

from oracle import np_oracle as npo

F32 = np.float32
ZN_TILE = 1024
WARP_ROW = 128        # 32 lanes x ZN_IPT = 4 points
SCAN_TILES = 8192     # 1024 threads x 8 tiles per round of k_zone_scan
SCAN_POINTS = SCAN_TILES * ZN_TILE
MAX_ZONES = 16
NOOP = (0, 1.0, 0.0, 1)   # negative stage with lo > hi: keeps every finite x, so it changes nothing in a chain
INF, FMAX = float("inf"), float(np.finfo(F32).max)


def np_zone_masks(x, zones) -> np.ndarray:
    """[n_zones, n] membership of every point (a zone without stages keeps every point)."""
    return np.array([npo.crop(x, chain) for chain in zones]).reshape(len(zones), len(x))


def with_noop(zones):
    """The same windows forced onto the chain path: the no-op stage appended to the first zone with room for it."""
    out = [list(z) for z in zones]
    for z in out:
        if 0 < len(z) < 4:
            z.append(NOOP)
            return out
    raise ValueError("no zone with room for the no-op stage")


def is_box(zones) -> bool:
    """derive_box: every zone has stages, none negative, no NaN limit."""
    return all(len(z) > 0 and all(not neg and lo == lo and hi == hi for (_, lo, hi, neg) in z) for z in zones)


def _index_cloud(n, seed=0):
    """x = the point's index (exact in float), so that windows on x cut at chosen indices; y in [0, 1)."""
    rng = np.random.default_rng(seed)
    x = np.zeros((n, 4), F32)
    x[:, 0] = np.arange(n, dtype=F32)
    x[:, 1] = rng.random(n).astype(F32)
    x[:, 2] = rng.uniform(-2, 2, n).astype(F32)
    x[:, 3] = rng.uniform(0, 255, n).astype(F32)
    x[3::11, 0] = -1.0 - x[3::11, 0]      # in no x window below
    return x


TILE_NS = (1, 31, 32, 127, 128, 129, 1023, 1024, 1025, 2049)
TILE_ZONES = [
    [(0, 0, 127, 0)], [(0, 128, 1023, 0)], [(0, 1024, 4096, 0)], [(0, 0, 1e9, 0)],     # warp-row and tile edges, all
    [(1, 0, 0.5, 0)], [(0, 31, 32, 0)], [(0, 127, 128, 0), (1, 0.25, 1, 0)], [(0, 1023, 1025, 0)],
    [(0, 0, 1e9, 0), (2, -1, 1, 0)], [(0, 0, 1e9, 0), (3, 0, 128, 0)], [(0, 2048, 2049, 0)], [(0, 1e6, 2e6, 0)],
    [(0, 64, 191, 0)], [(0, 896, 1151, 0)], [(1, 0.5, 1, 0), (0, 0, 1e9, 0)], [(0, 0, 1e9, 0), (2, -2, 2, 0)],
]
ONLY_15 = [[(0, 1e6, 2e6, 0)]] * 15 + [[(0, -1e9, 1e9, 0)]]
NESTED = [[(0, 64 * z + 64, 1e9, 0)] for z in range(MAX_ZONES)]   # x >= 1024: all 16 zones; starts at 128 and 1024


def tile_cases():
    cases = []
    for n in TILE_NS:
        x = _index_cloud(n, n)
        cases.append(dict(name="Z-tile:%d" % n, x=x, zones=TILE_ZONES))
        cases.append(dict(name="Z-tile:%d:nested" % n, x=x, zones=NESTED))
        cases.append(dict(name="Z-tile:%d:only15" % n, x=x, zones=ONLY_15))
    return cases


def path_cloud():
    """NaN and +-inf in each of x, y, z and intensity, +-0 against +-0 limits, +-FLT_MAX, values on the limits."""
    base = [-3.0, -1.0, -0.0, 0.0, 0.5, 1.0, 2.0, 3.0, FMAX, -FMAX]
    rows = []
    for a in base:
        for b in (-1.0, 0.0, -0.0, 1.0, 2.5):
            rows.append([a, b, -a, b * 10])
    bad = [float("nan"), INF, -INF]
    for ax in range(4):
        for v in bad:
            for b in (0.0, 1.0):
                r = [b, 0.5, -b, 7.0]
                r[ax] = v
                rows.append(r)
    return np.array(rows, F32)


PATH_SETS = {
    "basic": [[(0, -1, 1, 0)], [(1, 0, 2.5, 0), (3, 0, 10, 0)], [(2, -0.0, 0.0, 0)], [(0, 0.0, -0.0, 0)]],
    "inf-limits": [[(0, -INF, INF, 0)], [(1, -FMAX, FMAX, 0)], [(3, -INF, INF, 0)], [(2, -INF, 0, 0), (0, 0, INF, 0)]],
    "eq-and-empty": [[(0, 1, 1, 0)], [(1, 2.5, 2.5, 0)], [(0, 2, 1, 0)], [(3, 10, 10, 0), (0, -3, 3, 0)]],
    "two-stages-one-axis": [[(0, -2, 2, 0), (0, 0, 3, 0)], [(1, -1, 1, 0), (1, 0, 0, 0)], [(3, -10, 25, 0)]],
    "intensity": [[(3, -INF, INF, 0)], [(0, -INF, INF, 0)], [(3, 0, 10, 0), (1, -1, 1, 0)], [(2, -5, 5, 0)]],
    "negative": [[(0, -1, 1, 1)], [(1, 0, 1, 1), (0, -3, 3, 0)], [(3, 0, 10, 1)], [(2, 1, 0, 1)]],
    "nan-limits": [[(0, float("nan"), 1, 0)], [(1, 0, float("nan"), 0)], [(2, float("nan"), float("nan"), 1)],
                   [(3, float("nan"), 5, 0), (0, -3, 3, 0)]],
}


def path_cases():
    x = path_cloud()
    return [dict(name="Z-path:%s" % k, x=x, zones=z) for k, z in PATH_SETS.items()]


def scan_cloud(n, seed=1):
    """x = y = i % 16 (exact): zone z (x in [z, 100], y in [-100, z + 1]) holds the points with x in {z, z + 1}; the
    points at (100, -100) -- the first and last of every scan round, and every 100003rd -- are in all 16 zones."""
    rng = np.random.default_rng(seed)
    x = np.empty((n, 4), F32)
    x[:, 0] = (np.arange(n) % MAX_ZONES).astype(F32)
    x[:, 1] = x[:, 0]
    x[:, 2] = rng.random(n, dtype=np.float32)
    x[:, 3] = 1.0
    special = np.concatenate([np.arange(0, n, 100003), np.arange(0, n, SCAN_POINTS),
                              np.minimum(np.arange(1, n // SCAN_POINTS + 2) * SCAN_POINTS - 1, n - 1)])
    x[special, 0], x[special, 1] = 100.0, -100.0
    return x


SCAN_ZONES = [[(0, z, 100, 0), (1, -100, z + 1, 0)] for z in range(MAX_ZONES)]
SCAN_NS = (SCAN_POINTS + 1, 2 * SCAN_POINTS + 777)
KEEP_ALL = [[(0, -INF, INF, 0)]] * MAX_ZONES
GROW_NS = (ZN_TILE, ZN_TILE + 1, SCAN_POINTS + 1)
