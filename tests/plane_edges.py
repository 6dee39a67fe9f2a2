"""Edge inputs of the RANSAC ground plane (family P): cm_plane.cu's kernels and plane_ransac_run's host loop in cm_api.cu.

The constants below mirror the sources (tests/test_plane_edges.py pins each one to its source line). The cases sit on
the boundaries where the kernels and the host loop change what they do:
  - the scoring rounds of 32, 256 and then 1024 draws per cloud (cumulative edges 32, 288, 1312, 2336): P-batch;
  - getSamples' 1000 rejected draws in a row: P-bad;
  - k_plane_score's 512-point chunks, padded with NaN, and its 128-draw CTAs: P-chunk (a model with d = +-0, so that a
    zero-filled pad would be inside);
  - k_plane_moments' 256-point tiles, padded to whole groups of 32 terms, and the n_in < 4 refit floor: P-tile;
  - the strict `< threshold` of score, moments and select, and the float rounding of the double threshold: P-thr;
  - probability, iteration cap and seed extremes: P-settings; eight-cloud layouts and mask bits 2k / 2k + 1: P-multi;
  - clouds past one and two rounds of k_zone_scan's 8192-tile loop in the given-mask compaction: P-size.

A case is a dict: clouds (list of float32 [n, 4]), threshold, probability, max_iterations, seed, orders (the sum orders
it runs), optimizes (the refit settings it runs), plus what the CPU tests check about it."""
from __future__ import annotations

import numpy as np

F32 = np.float32

PL_THREADS = 128       # k_plane_score: draws per CTA
PL_CHUNK = 512         # k_plane_score: points per CTA, NaN-padded
PM_TILE = 256          # k_plane_moments: points per tile
PM_STRIDE = 276        # k_plane_moments: staged row length (the tile + the adding warp's prefetch slack)
SELECT_BLOCK = 256     # k_plane_select: points per CTA
FIRST_BATCH, SECOND_BATCH, BATCH = 32, 256, 1024   # PLANE_FIRST_BATCH / PLANE_SECOND_BATCH / PLANE_BATCH
REJECT_LIMIT = 1000    # getSamples' max_sample_checks_: ++s.bad_run == 1000
REFIT_FLOOR = 4        # optimizeModelCoefficients needs n_in >= 4
MAX_CLOUDS = 8         # CM_MAX_PLANE_CLOUDS
ZONE_LAUNCHES = 3      # CM_ZONE_LAUNCHES: count, scan, scatter (the scan alone without points)
SCAN_ROUND = 1024 * 8 * 1024   # points per round of k_zone_scan's tile loop (8192 tiles of 1024)

EDGES = (32, 288, 1312, 2336)   # cumulative draws at the end of rounds 1 .. 4


def round_sizes(rounds: int) -> list:
    return [FIRST_BATCH if r == 0 else SECOND_BATCH if r == 1 else BATCH for r in range(rounds)]


def round_of_draw(d: int) -> int:
    """The scoring round (1-based) that holds a cloud's d-th draw; 0 for no draws."""
    if d <= 0:
        return 0
    r, end = 0, 0
    while end < d:
        end += round_sizes(r + 1)[-1]
        r += 1
    return r


def plane_rounds(draws_per_cloud) -> int:
    """Scoring rounds of one call: the round holding each cloud's last draw, maximised over the clouds."""
    return max([round_of_draw(int(d)) for d in draws_per_cloud] + [0])


def plane_launches(draws_per_cloud, optimize: bool, any_found: bool, n_points: int) -> int:
    """cm_launch_count after a plane call: a k_plane_score per round, k_plane_moments when a model is refitted, a
    k_plane_select when there are points, and the given-mask zone split (count, scan, scatter; the scan alone without
    points)."""
    return (plane_rounds(draws_per_cloud) + (1 if optimize and any_found else 0) + (1 if n_points else 0)
            + (ZONE_LAUNCHES if n_points else 1))


class _Shuffle:
    """SampleConsensusModel::shuffled_indices_ as a sparse map (identity where no swap has touched it)."""

    def __init__(self):
        self.m = {}

    def get(self, i):
        return self.m.get(i, i)

    def swap(self, a, b):
        va, vb = self.get(a), self.get(b)
        self.m[a], self.m[b] = vb, va


def draw_stream(n: int, seed: int, count: int) -> np.ndarray:
    """The first `count` three-index draws of PCL's sampler on a cloud of n points: mt19937(seed) >> 1 (boost's
    uniform_int over [0, INT_MAX]), then a partial Fisher-Yates shuffle of the first three positions. Independent of
    the data: a rejected draw is drawn again from the same stream."""
    assert n >= 3
    raw = np.random.RandomState(seed & 0xFFFFFFFF)._bit_generator.random_raw(3 * count).astype(np.uint64) >> np.uint64(1)
    sh = _Shuffle()
    out = np.empty((count, 3), np.int64)
    for d in range(count):
        for i in range(3):
            sh.swap(i, i + int(raw[3 * d + i]) % (n - i))
        out[d] = (sh.get(0), sh.get(1), sh.get(2))
    return out


def _generic(n, seed, scale=20.0):
    """Points in general position: no draw of three is collinear."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-scale, scale, (n, 4)).astype(F32)
    x[:, 3] = rng.uniform(0, 255, n).astype(F32)
    return x


def ground(n, seed, frac, noise=0.03, slope=0.02):
    rng = np.random.default_rng(seed)
    g = int(round(n * frac))
    x = np.zeros((n, 4), F32)
    x[:, 0] = rng.uniform(-30, 30, n)
    x[:, 1] = rng.uniform(-10, 10, n)
    x[:g, 2] = -1.8 + slope * x[:g, 0] + rng.normal(0, noise, g)
    x[g:, 2] = rng.uniform(-1.5, 1.0, n - g)
    x[:, 3] = rng.uniform(0, 255, n)
    return x[rng.permutation(n)]


def _case(name, clouds, thr=0.3, prob=0.99, max_it=1000, seed=12345, orders=(0,), optimizes=(False, True), **kw):
    d = dict(name=name, clouds=[np.ascontiguousarray(c, F32) for c in clouds], threshold=float(thr),
             probability=float(prob), max_iterations=int(max_it), seed=int(seed), orders=tuple(orders),
             optimizes=tuple(optimizes))
    d.update(kw)
    return d


# ---- P-batch ------------------------------------------------------------------------------------------------------------
# (inlier share, seed) found by a seed search on the CPU (tests/test_plane_edges.py re-derives the iteration counts):
# with k_cloud(share) at probability 0.99
# the stopping rule ends exactly at these iterations, one on and one past the first and second round edges
K_STOP_SEEDS = {32: (0.5, 97), 33: (0.5, 1), 288: (0.22, 1898), 289: (0.24, 3213)}


def k_cloud(frac, n=1500, seed=77):
    """Ground (noise well inside the threshold) and outliers spread over 20 m of height: the inlier share is ~frac."""
    x = ground(n, seed, frac, noise=0.05)
    off = np.abs(x[:, 2] + 1.8 - 0.02 * x[:, 0]) > 0.25
    x[off, 2] = np.random.default_rng(seed + 1).uniform(-10, 10, int(off.sum())).astype(F32)
    return x


def batch_cases():
    cases = []
    cloud = _generic(200, 1)
    for b in EDGES:
        for m in (b - 2, b - 1, b):
            cases.append(_case("P-batch:cap:%d" % m, [cloud], prob=1.0, max_it=m, orders=(0,), optimizes=(False,),
                               draws=m + 1))
    for it, (frac, seed) in K_STOP_SEEDS.items():
        cases.append(_case("P-batch:k:%d" % it, [k_cloud(frac)], seed=seed, orders=(0, 1, 2), iterations=it))
    return cases


# ---- P-bad --------------------------------------------------------------------------------------------------------------
BAD_N = 20000


def bad_cloud(first_good: int, seed: int = 12345, n: int = BAD_N, extra: int = 40):
    """An exactly collinear line (t, 2t, 4t, t) with integer t, except at off-line indices chosen from the draw stream:
    no draw before `first_good` touches one (every one of them is rejected) and draw `first_good` does."""
    s = draw_stream(n, seed, first_good)
    before = set(s[:-1].ravel().tolist())
    hit = [int(i) for i in s[-1] if int(i) not in before]
    assert hit, "draw %d of seed %d has no fresh index" % (first_good, seed)
    t = np.arange(n, dtype=F32)
    x = np.column_stack([t, 2 * t, 4 * t, t]).astype(F32)
    rng = np.random.default_rng(first_good)
    free = np.setdiff1d(np.arange(n), np.array(sorted(before | set(s[-1].tolist())), np.int64))
    off = np.array([hit[0]] + rng.choice(free, extra, replace=False).tolist(), np.int64)
    x[off, 0] += F32(3.0)
    x[off, 2] -= F32(5.0)
    return x, off


def bad_cases():
    cases = []
    for d in (33, 289, REJECT_LIMIT, REJECT_LIMIT + 1):   # at 1001 getSamples has given up after draw 1000
        x, off = bad_cloud(d)
        cases.append(_case("P-bad:%d" % d, [x], thr=0.5, orders=(0,), optimizes=(False, True), first_good=d, off=off))
    return cases


# ---- P-chunk ------------------------------------------------------------------------------------------------------------
CHUNK_NS = (3, 4, 127, 128, 129, 511, 512, 513, 1023, 1024, 1025, 1537)


def chunk_cloud(n, offset=0.0, seed=0):
    """Ground exactly on z = offset (d = +-0 at offset 0: a zero-filled pad point would be inside), a quarter of the
    points 2 m above; ground points sit at indices 511 / 512 and 1023 / 1024 where the cloud reaches them."""
    rng = np.random.default_rng(1000 + n + seed)
    x = np.zeros((n, 4), F32)
    x[:, 0] = rng.uniform(-20, 20, n)
    x[:, 1] = rng.uniform(-20, 20, n)
    x[:, 2] = F32(offset)
    up = rng.random(n) < 0.25
    up[[i for i in (0, 1, 2, 511, 512, 1023, 1024) if i < n]] = False
    x[up, 2] = F32(offset + 2.0)
    x[:, 3] = rng.uniform(0, 255, n)
    return x


def chunk_cases():
    cases = []
    for n in CHUNK_NS:
        cases.append(_case("P-chunk:%d" % n, [chunk_cloud(n)], orders=(0, 1, 2), optimizes=(False, True), zero_d=True))
        cases.append(_case("P-chunk:%d:offset" % n, [chunk_cloud(n, 1.5)], orders=(0,), optimizes=(False, True)))
    # a noisy plane through the origin: a zero-filled pad point of k_plane_moments would join the refit sums and count
    rng = np.random.default_rng(5)
    for n in (200, 300, 1000):
        x = np.zeros((n, 4), F32)
        x[:, :2] = rng.uniform(-20, 20, (n, 2))
        x[:, 2] = (0.1 * x[:, 0] - 0.05 * x[:, 1] + rng.normal(0, 0.02, n)).astype(F32)
        x[:, 3] = 1.0
        cases.append(_case("P-chunk:origin:%d" % n, [x], orders=(0, 1, 2), optimizes=(True,)))
    return cases


# ---- P-tile -------------------------------------------------------------------------------------------------------------
TILE_COUNTS = (0, 1, 15, 16, 17, 31, 32, 33, 63, 64, 65, 255, 256)
TILE_NORMAL = (0.03, -0.02)   # z = 0.03 (x - 1000) - 0.02 (y - 1000) + 1000: tilted, near 1000 m


def tile_cloud(n, counts, seed=0, first_last=True):
    """Tiles of PM_TILE points; tile t holds counts[t] inliers on the tilted plane (noise-free to float rounding), the
    rest 20 .. 60 m above or below it. first_last: inliers at the first and last index of every tile that has two."""
    rng = np.random.default_rng(seed)
    x = np.zeros((n, 4), F32)
    x[:, 0] = (1000.0 + rng.uniform(-40, 40, n)).astype(F32)
    x[:, 1] = (1000.0 + rng.uniform(-40, 40, n)).astype(F32)
    plane = 1000.0 + TILE_NORMAL[0] * (x[:, 0].astype(np.float64) - 1000.0) + TILE_NORMAL[1] * (x[:, 1].astype(np.float64) - 1000.0)
    inl = np.zeros(n, bool)
    for t in range((n + PM_TILE - 1) // PM_TILE):
        a, b = t * PM_TILE, min(n, (t + 1) * PM_TILE)
        k = min(counts[t % len(counts)], b - a)
        if k == 0:
            continue
        if k == b - a:
            pick = np.arange(a, b)
        elif first_last and k >= 2:
            pick = np.concatenate([[a, b - 1], rng.choice(np.arange(a + 1, b - 1), k - 2, replace=False)])
        else:
            pick = rng.choice(np.arange(a, b), k, replace=False)
        inl[pick] = True
    sign = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    z = np.where(inl, plane, plane + sign * rng.uniform(20, 60, n))
    x[:, 2] = z.astype(F32)
    x[:, 3] = rng.uniform(0, 255, n).astype(F32)
    return x, inl


def tile_cases():
    cases = []
    for n in (255, 256, 257, 511, 512, 513, 2000):
        counts = [c for c in TILE_COUNTS]
        rng = np.random.default_rng(n)
        counts = list(rng.permutation(counts)) if n > 600 else [max(c, 64) for c in counts[::3]]
        x, inl = tile_cloud(n, counts, seed=n)
        cases.append(_case("P-tile:%d" % n, [x], prob=0.999, orders=(0, 1, 2), optimizes=(True,), inliers=inl))
    # every per-tile count of TILE_COUNTS once, an all-outlier tile between inlier tiles
    counts = [200, 0] + list(TILE_COUNTS) + [0, 256]
    x, inl = tile_cloud(PM_TILE * len(counts), counts, seed=99)
    cases.append(_case("P-tile:counts", [x], prob=0.999, orders=(0, 1, 2), optimizes=(True,), inliers=inl,
                       tile_counts=counts))
    for k in (3, 4, 5):   # exactly 3, 4 and 5 inliers: the refit floor
        x, inl = tile_cloud(12, [k], seed=k + 2, first_last=False)
        cases.append(_case("P-tile:floor:%d" % k, [x], thr=0.01, prob=0.99, max_it=1000, orders=(0, 1, 2), optimizes=(True,),
                           inliers=inl, floor=k))
    return cases


# ---- P-thr --------------------------------------------------------------------------------------------------------------
def _f32_up(v):
    return float(np.nextafter(F32(v), F32(np.inf)))


def _f32_down(v):
    return float(np.nextafter(F32(v), F32(-np.inf)))


FMAX = float(np.finfo(F32).max)
TINY = float(np.nextafter(F32(0), F32(1)))   # the smallest float subnormal
THRESHOLDS = {
    "0.25": 0.25,                                 # a float
    "0.3": 0.3,                                   # float(0.3) rounds up
    "0.3f+ulp": float(np.nextafter(np.float64(F32(0.3)), np.inf)),   # float(thr) rounds down: the nextafter decides
    "0": 0.0,
    "subnormal": TINY,
    "dsubnormal": 5e-324,                         # the smallest double subnormal: every float 0 is inside
    "fmax": FMAX,
    "1e300": 1e300,                               # above FLT_MAX
    "inf": float("inf"),
    "-inf": float("-inf"),
    "nan": float("nan"),
    "-1": -1.0,
}


def effective_threshold(thr: float):
    """The float the kernels compare with: the smallest float >= the double threshold (inf above FLT_MAX)."""
    if thr > FMAX:
        return F32(np.inf)
    with np.errstate(over="ignore"):
        t = F32(thr)
    if np.float64(t) < thr:
        t = np.nextafter(t, F32(np.inf))
    return t


def thr_points(thr):
    """z values at +-t, +-nextbelow(t), +-nextabove(t) for t = the float nearest the threshold, and +-0."""
    if not np.isfinite(thr) or thr < 0:
        t = F32(0.3)
    else:
        with np.errstate(over="ignore"):
            t = F32(min(thr, FMAX))
    with np.errstate(over="ignore"):
        vals = [t, np.nextafter(t, F32(-np.inf)), np.nextafter(t, F32(np.inf))]
    zs = []
    for v in vals:
        if np.isfinite(v):
            zs += [v, -v]
    zs += [F32(0.0), F32(-0.0)]
    return np.array(zs, F32)


def thr_cloud(thr, n_ground=300, seed=3):
    rng = np.random.default_rng(seed)
    zs = thr_points(thr)
    x = np.zeros((n_ground + len(zs), 4), F32)
    x[:, 0] = rng.uniform(-10, 10, len(x))
    x[:, 1] = rng.uniform(-10, 10, len(x))
    x[n_ground:, 2] = zs
    x[:, 3] = 7.0
    return x, n_ground


def thr_cases():
    cases = []
    for name, thr in THRESHOLDS.items():
        x, g = thr_cloud(thr)
        cases.append(_case("P-thr:%s" % name, [x], thr=thr, prob=1.0, max_it=20, orders=(0, 1, 2),
                           optimizes=(False, True), thr_from=g))
    return cases


# ---- P-settings ---------------------------------------------------------------------------------------------------------
def settings_cases():
    cases = []
    g = ground(3000, 8, 0.6)
    for p in (0.0, 1.0, float("nan"), 1.5):
        cases.append(_case("P-settings:prob:%r" % p, [g], prob=p, max_it=300, orders=(0,), optimizes=(False, True)))
    cases.append(_case("P-settings:max_it:0", [g], max_it=0, orders=(0,), optimizes=(False, True)))
    for s in (0, 1, 2**32 - 1):
        cases.append(_case("P-settings:seed:%d" % s, [g], seed=s, orders=(0,), optimizes=(False, True)))
    cases.append(_case("P-settings:long", [ground(20000, 9, 0.5)], prob=1.0, max_it=5000, orders=(0,),
                       optimizes=(True,), big=True))
    return cases


# ---- P-multi ------------------------------------------------------------------------------------------------------------
def multi_cases():
    t = np.arange(60, dtype=F32)
    line = np.column_stack([t, 2 * t, 4 * t, t]).astype(F32)
    e = np.zeros((0, 4), F32)
    cases = []
    # cloud boundaries off the 256-point select blocks and 1024-point zone tiles; cloud 7 non-empty (mask bits 14, 15)
    sizes = (1000, 300, 1500, 77, 2600, 513, 1029, 999)
    cases.append(_case("P-multi:offgrid", [ground(s, 200 + i, 0.7) for i, s in enumerate(sizes)],
                       orders=(0, 1, 2), optimizes=(False, True)))
    cases.append(_case("P-multi:empties", [e, ground(700, 210, 0.7), e, e, ground(1300, 211, 0.6), e,
                                           ground(257, 212, 0.8), e], orders=(0,), optimizes=(False, True)))
    cases.append(_case("P-multi:tiny", [ground(1, 220, 1.0), ground(2, 221, 1.0), ground(3, 222, 1.0), line,
                                        ground(900, 223, 0.7), e, ground(4, 224, 1.0), ground(1100, 225, 0.7)],
                       orders=(0,), optimizes=(False, True)))
    # clouds whose stopping rule ends in rounds 1, 2, 3 and 4 of the same call: later rounds score only some clouds
    fr = (0.9, 0.35, 0.14, 0.08, 0.9, 0.35, 0.12, 0.08)
    cases.append(_case("P-multi:rounds", [k_cloud(f, 700 + 91 * i, 240 + i) for i, f in enumerate(fr)], max_it=3000,
                       orders=(0,), optimizes=(False, True), rounds=(1, 2, 3, 4)))
    return cases


def size_cases():
    """One cloud just past one scan round (8388609 points) and eight clouds just past two (2 x 8388608 + 777)."""
    n1 = SCAN_ROUND + 1
    n8 = 2 * SCAN_ROUND + 777
    per = [n8 // 8 + (1 if i < n8 % 8 else 0) for i in range(8)]
    return [_case("P-size:one", [ground(n1, 300, 0.8)], orders=(0,), optimizes=(True,)),
            _case("P-size:eight", [ground(p, 310 + i, 0.75) for i, p in enumerate(per)], orders=(0,), optimizes=(True,))]


def plane_cases(with_size: bool = False) -> dict:
    out = {}
    for c in batch_cases() + bad_cases() + chunk_cases() + tile_cases() + thr_cases() + settings_cases() + multi_cases():
        out[c["name"]] = c
    if with_size:
        for c in size_cases():
            out[c["name"]] = c
    return out
