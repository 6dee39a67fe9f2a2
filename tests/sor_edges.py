"""Edge inputs of the statistical outlier removal (family S) and a numpy restatement of its plan and search -- TEST
INFRASTRUCTURE ONLY.

sor_plan restates the host side of statistical_outlier_run (cm_api.cu): sor_cell_edge (double arithmetic, the largest
cloud by finite count, the key-range floor, the clamps), inv = f32(1.0 / edge), every cloud's grid as k_grid_setup forms
it with that inv, the key plan (frame bits with the sentinel frame of non-finite points, idx_bits, key bytes, radix
passes), the direct-address table and the launch count cm_launch_count reports. sor_search restates k_sor_knn's search:
the growing cubes of cells, its stopping rule and the row pieces it visits. sum_path restates k_sor_sums' exactness
condition. The constants mirror the sources; test_sor_edges.py reads them out of them.

Families (sor_cases()):
  S-slots   mean_k around the register-slot rows (NS = 1 / 2 / 4), exactly mean_k + 1 finite points, cells whose
            occupancy makes one batch of 32 candidates fill the slots across a 32-slot row;
  S-bound   the deciding neighbour just past the cube of half-width r, through faces, edges and corners, in clipped
            cubes, near the origin and at |x * inv| ~ 2^19 where fl(x * inv) rounds a point across a cell plane;
  S-plan    key widths 32 / 33 bits and 1 ... 8 radix passes, the sentinel frame, the table limit 2^25, the key-range
            floor through magnitude and extent, the clamps 1e-30 and 1e36;
  S-sums    both sums just below and just above 2^(53 + e_min), subnormal and overflowing values, the SUM_THREADS and
            SERIAL_TILE strides, 16 clouds on different paths;
  S-select  distances equal to the threshold, empty clouds first, in the middle and last."""
from __future__ import annotations

import math

import numpy as np

import sor_np

F32 = np.float32

# ---- constants of cm_statistical.cu / cm_api.cu / cm_voxel.cu ----------------------------------------------------------
SOR_NS_LIMITS = (32, 64)          # mean_k + 1 <= 32: one slot per lane (NS = 1), <= 64: NS = 2, otherwise NS = 4
SOR_WARPS = 8                     # warps (points) per CTA of k_sor_knn
SUM_THREADS = 1024                # CTA of k_sor_sums (the stride of its parallel pass)
SERIAL_TILE = 4096                # values per shared-memory tile of the serial chain
EPS_REL = 2.0 ** -23              # eps = (M * EPS_REL * EPS_MARGIN + EPS_ABS) cells, M = max(|min_b|, |max_b|) + 1
EPS_MARGIN = 1.0 + 2.0 ** -20
EPS_ABS = 2.0 ** -140
BOUND_FACTOR = 1.0 - 2.0 ** -20   # B = ((r - eps) * h)^2 * BOUND_FACTOR, used only when B >= BOUND_FLOOR
BOUND_FLOOR = 2.0 ** -100
FLOOR_MAG = 2.0 ** 20             # key-range floor of the edge: |x| / edge <= 2^20 and extent / edge <= 2^19 ...
FLOOR_EXTENT = 2.0 ** 19
FLOOR_MARGIN = 1.0 + 1.0 / 1024.0  # ... times this margin
EDGE_MIN, EDGE_MAX = 1e-30, 1e36  # 1 / edge stays a normal float
TABLE_LOG2 = 25                   # the table is used while n_clouds << idx_bits <= 2^25
RADIX_BITS = 8
MAX_PASSES = 8
GRID_RANGE_CELLS = 1 << 21        # k_grid_setup: more cells on an axis, or a coordinate beyond 2^30 cells, is out of range
GRID_RANGE_ORIGIN = 1 << 30

# Cost guard of the GPU cases, in row pieces (one table or binary-search lookup pair each; a warp takes 32 at a time).
# The 58 k ROI at mean_k 10 visits about 3.5 M pieces in 0.34 ms of kNN on a B200 (DESIGN section 8). A point's pieces
# run serially in its warp; the worst point of a case may take 2^23 pieces and a case 2^31 in all. The cases use at most
# 3.5 M pieces per point and 7 M per call; all 90 of test_gpu_sor_edges.py ran in 5.3 s on a B200 at 1000 W.
COST_WORST = 1 << 23
COST_TOTAL = 1 << 31


def ns_of(mean_k: int) -> int:
    return 1 if mean_k + 1 <= SOR_NS_LIMITS[0] else 2 if mean_k + 1 <= SOR_NS_LIMITS[1] else 4


def next_r(r: int) -> int:
    return r + max(1, r >> 1)


def growth(limit: int = 1 << 22) -> list:
    """the half-widths k_sor_knn visits: 0, 1, 2, 3, 4, 6, 9, 13, 19, 28, ..."""
    out, r = [], 0
    while r <= limit:
        out.append(r)
        r = next_r(r)
    return out


def _bits(cells: int) -> int:
    return 0 if cells <= 1 else int(cells - 1).bit_length()


def _fin(c) -> np.ndarray:
    return np.isfinite(np.asarray(c, F32)[:, :3]).all(axis=1)


# ---- the plan ----------------------------------------------------------------------------------------------------------
def sor_cell_edge(clouds, mean_k: int, forced_cell=None) -> dict:
    """sor_cell_edge of cm_api.cu. Returns the edge and its parts: the estimate (or the forced edge), the floor times its
    margin, and whether a clamp bound it."""
    floor_edge, edge, biggest = 0.0, 1.0, 0
    for c in clouds:
        c = np.asarray(c, F32).reshape(-1, 4)
        fin = _fin(c)
        n = int(fin.sum())
        if n <= 0:
            continue
        mn = c[fin, :3].min(axis=0).astype(np.float64)
        mx = c[fin, :3].max(axis=0).astype(np.float64)
        e = [float(mx[a]) - float(mn[a]) for a in range(3)]
        for a in range(3):
            mag = max(abs(float(mn[a])), abs(float(mx[a])))
            floor_edge = max(floor_edge, max(mag / FLOOR_MAG, e[a] / FLOOR_EXTENT))
        e.sort(reverse=True)
        ec = 1.0
        if e[1] > 0.0:
            ec = math.sqrt((mean_k + 1.0) * e[0] * e[1] / (3.141592653589793 * float(n)))
        elif e[0] > 0.0:
            ec = (mean_k + 1.0) * e[0] / (2.0 * float(n))
        if n > biggest:
            biggest, edge = n, ec
    if forced_cell is not None and float(forced_cell) > 0.0:
        edge = float(forced_cell)
    estimate = edge
    floored = floor_edge * FLOOR_MARGIN
    edge = max(edge, floored)
    out = min(max(edge, EDGE_MIN), EDGE_MAX)
    return dict(edge=out, estimate=estimate, floor=floored, floor_binds=floored > estimate,
                clamp=("min" if edge < EDGE_MIN else "max" if edge > EDGE_MAX else None))


def cells_of(xyz, inv) -> np.ndarray:
    """floor(f32(x * inv)) per coordinate (float64 array)."""
    with np.errstate(over="ignore", invalid="ignore"):
        return np.floor((np.asarray(xyz, F32)[:, :3] * F32(inv)).astype(F32)).astype(np.float64)


def sor_grid(x, inv) -> dict:
    """k_grid_setup of one cloud with the statistical removal's inv: min_b, max_b, div_b, zero_keys, index bits."""
    x = np.asarray(x, F32).reshape(-1, 4)
    fin = _fin(x)
    if not fin.any():
        z = np.zeros(3, np.int64)
        return dict(empty=True, min_b=z, max_b=z, div=z, zero_keys=False, bits=0)
    fc = cells_of(x[fin], inv)
    fmn, fmx = fc.min(axis=0), fc.max(axis=0)
    err = bool((np.abs(fmn) >= GRID_RANGE_ORIGIN).any() or (np.abs(fmx) >= GRID_RANGE_ORIGIN).any())
    lim = float(2 ** 31 - 1)
    mn = np.clip(fmn, -lim - 1, lim).astype(np.int64)
    mx = np.clip(fmx, -lim - 1, lim).astype(np.int64)
    div = mx - mn + 1
    err = err or bool((div > GRID_RANGE_CELLS).any())
    cells = 1 if err else int(div[0]) * int(div[1]) * int(div[2])
    return dict(empty=False, min_b=mn, max_b=mx, div=div, zero_keys=err, bits=_bits(cells))


def sor_plan(clouds, mean_k: int, forced_cell=None, table: bool = True) -> dict:
    """The plan of one statistical_outlier_multi call (a single cloud is a list of one); table=False is CM_SOR_NO_TABLE."""
    clouds = [np.asarray(c, F32).reshape(-1, 4) for c in clouds]
    n = len(clouds)
    ce = sor_cell_edge(clouds, mean_k, forced_cell)
    inv = F32(1.0 / ce["edge"])
    grids = [sor_grid(c, inv) for c in clouds]
    has_invalid = any((~_fin(c)).any() for c in clouds)
    frame_bits = _bits(n + (1 if has_invalid else 0))
    idx_bits = max([g["bits"] for g in grids if not g["empty"]] + [0])
    total = frame_bits + idx_bits
    key_range = any(g["zero_keys"] for g in grids) or total > 64
    total = min(total, 64)
    idx_bits = total - frame_bits
    passes = max(1, -(-total // RADIX_BITS))
    n_points = sum(len(c) for c in clouds)
    use_table = table and n_points > 0 and idx_bits <= TABLE_LOG2 and (n << idx_bits) <= (1 << TABLE_LOG2)
    # cm_launch_count: a bounding box per non-empty cloud, grid setup, keys, the radix passes, the table when used,
    # gather + kNN, sums + select (the zone compaction counts in its own workspace)
    launches = sum(1 for c in clouds if len(c)) + 2 + passes + (1 if use_table else 0) + 2 + 2
    return dict(edge=ce["edge"], estimate=ce["estimate"], floor=ce["floor"], floor_binds=ce["floor_binds"],
                clamp=ce["clamp"], inv=inv, cell=1.0 / float(inv), grids=grids, has_invalid=has_invalid,
                frame_bits=frame_bits, idx_bits=idx_bits, total_bits=total, key_bytes=4 if total <= 32 else 8,
                passes=passes, table=use_table, table_keys=(n << idx_bits) if use_table else 0, key_range=key_range,
                launches=launches)


# ---- the search --------------------------------------------------------------------------------------------------------
def search_eps(grid) -> float:
    mb = int(max(np.abs(grid["min_b"]).max(), np.abs(grid["max_b"]).max()))
    return (float(mb) + 1.0) * EPS_REL * EPS_MARGIN + EPS_ABS


def bound_at(r: int, eps: float, cell: float) -> float:
    """k_sor_knn's bound after the cube of half-width r (0 where it does not apply)."""
    m = float(r) - eps
    if not m > 0.0:
        return 0.0
    a = m * cell
    b = a * a * BOUND_FACTOR
    return b if b >= BOUND_FLOOR else 0.0


def sor_search(cloud, plan, mean_k: int, eps_scale: float = 1.0, frame: int = 0, chunk: int = 128) -> dict:
    """k_sor_knn for the finite points of one cloud (frame `frame` of the plan), vectorised over points; meant for clouds
    of a few thousand points (it forms every pair). Per finite point, in input order: "stop" (the half-width at which the
    search ends), "knn" (the mean_k + 1 kept float squared distances, ascending) and "pieces" (row pieces visited: 2 * rows
    of every cube, the kernel's cost). eps_scale scales the bound's eps (0: a kernel without it)."""
    x = np.asarray(cloud, F32).reshape(-1, 4)
    p = np.ascontiguousarray(x[_fin(x), :3])
    n, kp1 = len(p), mean_k + 1
    g = plan["grids"][frame]
    cells = (cells_of(p, plan["inv"]) - g["min_b"]).astype(np.int64)
    div = g["div"].astype(np.int64)
    eps = search_eps(g) * eps_scale
    cell = plan["cell"]
    stop = np.full(n, -1, np.int64)
    pieces = np.zeros(n, np.int64)
    knn = np.zeros((n, kp1), F32)
    if n < kp1:
        return dict(stop=stop, knn=knn, pieces=pieces)
    for s in range(0, n, chunk):
        q, cq = p[s:s + chunk], cells[s:s + chunk]
        D = np.abs(cq[:, None, :] - cells[None, :, :]).max(axis=2)
        dist = sor_np._sq_dist(q, p[None, :, :])
        act = np.arange(len(q))
        r = 0
        while len(act):
            c = cq[act]
            lo = np.maximum(c - r, 0)
            hi = np.minimum(c + r, div - 1)
            pieces[s + act] += 2 * (hi[:, 2] - lo[:, 2] + 1) * (hi[:, 1] - lo[:, 1] + 1)
            covers = (lo == 0).all(axis=1) & (hi == div - 1).all(axis=1)
            inside = D[act] <= r
            full = inside.sum(axis=1) >= kp1
            vals = np.where(inside, dist[act], F32(np.inf))
            part = np.sort(vals, axis=1)[:, :kp1]
            kth = part[:, -1].astype(np.float64)
            b = bound_at(r, eps, cell)
            done = covers | (full & (kth <= 0.0)) | (full & (b > 0.0) & (b >= kth))
            stop[s + act[done]] = r
            knn[s + act[done]] = part[done]
            act = act[~done]
            r = next_r(r)
    return dict(stop=stop, knn=knn, pieces=pieces)


def search_cost(clouds, plan, mean_k: int) -> tuple:
    """(worst, total) row pieces of a call: every cloud that is not too few for mean_k."""
    worst = total = 0
    for f, c in enumerate(clouds):
        nf = int(_fin(c).sum())
        if nf <= mean_k:
            continue
        pc = sor_search(c, plan, mean_k, frame=f)["pieces"]
        worst, total = max(worst, int(pc.max())), total + int(pc.sum())
    return worst, total


# ---- the sums ----------------------------------------------------------------------------------------------------------
def lsb_exp(v) -> np.ndarray:
    """exponent of the lowest set bit of every non-negative float32 (a large value for 0), as k_sor_sums' lsb_exp."""
    b = np.asarray(v, F32).view(np.uint32).astype(np.int64) & 0x7FFFFFFF
    ex, man = b >> 23, b & 0x7FFFFF
    full = np.where(ex > 0, man | 0x800000, man)
    low = full & -full
    tz = np.where(low > 0, np.log2(np.maximum(low, 1)).astype(np.int64), 0)
    out = np.where(ex > 0, ex - 150 + tz, -149 + tz)
    return np.where(b == 0, 1 << 30, out)


def sum_path(dist, force: bool = False) -> int:
    """k_sor_sums' path: bit 0 the sum, bit 1 the sum of float squares runs PCL's serial chain. A sum is taken in parallel
    iff every value is finite and non-negative and the exact total is below 2^(53 + e_min)."""
    v = np.asarray(dist, F32)
    with np.errstate(over="ignore"):
        v2 = (v * v).astype(F32)
    path = 3 if force else 0
    for bit, w in ((1, v), (2, v2)):
        if not len(w):
            continue
        if (~np.isfinite(w)).any() or (w < 0).any():
            path |= bit
            continue
        e = int(lsb_exp(w).min())
        if e < (1 << 30) and not math.fsum(w.astype(np.float64).tolist()) < math.ldexp(1.0, 53 + e):
            path |= bit
    return path


# ---- S-slots -----------------------------------------------------------------------------------------------------------
SLOT_MEAN_KS = (30, 31, 32, 33, 62, 63, 64, 65, 126)
SLOT_EXACT_KS = (31, 32, 63, 64, 126)
SLOT_CELL_COUNTS = (20, 45, 50, 70)


def _xyzi(xyz) -> np.ndarray:
    xyz = np.asarray(xyz, F32).reshape(-1, 3)
    return np.ascontiguousarray(np.column_stack([xyz, np.zeros(len(xyz), F32)]))


def slot_lattice(mean_k: int) -> np.ndarray:
    """a cubic lattice big enough that interior points have mean_k + 1 neighbours with ties at the k-th distance."""
    side = 7 if mean_k < 64 else 9
    g = np.arange(side, dtype=F32) * F32(0.25)
    x, y, z = np.meshgrid(g, g, g, indexing="ij")
    return _xyzi(np.column_stack([x.ravel(), y.ravel(), z.ravel()]))


def slot_blob(seed: int, n: int = 1500) -> np.ndarray:
    rng = np.random.default_rng(seed)
    return _xyzi(rng.normal(scale=0.6, size=(n, 3)))


def slot_exact(mean_k: int, seed: int = 0) -> np.ndarray:
    """exactly mean_k + 1 finite points and three non-finite rows."""
    rng = np.random.default_rng(seed + mean_k)
    c = _xyzi(rng.uniform(-1, 1, (mean_k + 1, 3)))
    bad = np.array([[np.nan, 0, 0, 0], [0, np.inf, 0, 0], [0, 0, -np.inf, 0]], F32)
    out = np.concatenate([c[: mean_k // 2], bad[:2], c[mean_k // 2:], bad[2:]])
    return np.ascontiguousarray(out)


SLOT_CELL = 1.0


def slot_cells(seed: int = 0) -> np.ndarray:
    """a 3 x 3 x 3 block of unit cells (forced edge SLOT_CELL) whose occupancies cycle through SLOT_CELL_COUNTS: the
    search of a point in a cell of 20 (45, 50, 70) takes that many candidates at r = 0 and then a first batch of 32 at
    r = 1, which fills the slots across the 32- (64-) slot row."""
    rng = np.random.default_rng(seed)
    pts = []
    for k, (i, j, l) in enumerate(np.ndindex(3, 3, 3)):
        m = SLOT_CELL_COUNTS[k % len(SLOT_CELL_COUNTS)]
        pts.append(np.array([i, j, l], np.float64) + rng.uniform(0.05, 0.95, (m, 3)))
    return _xyzi(np.concatenate(pts))


def fill_crossings(cloud, plan, mean_k: int) -> int:
    """points whose first candidate batch at r = 1 fills slots from below a multiple of 32 to above it: r = 0 takes the
    own cell (filled = min(own, kp1), batches of 32), r = 1 (18 pieces: one round) then takes min(32, candidates)."""
    x = np.asarray(cloud, F32)
    p = x[_fin(x)]
    g = plan["grids"][0]
    c = (cells_of(p, plan["inv"]) - g["min_b"]).astype(np.int64)
    kp1 = mean_k + 1
    cnt = 0
    for i in range(len(p)):
        d = np.abs(c - c[i]).max(axis=1)
        own, ring = int((d == 0).sum()), int((d == 1).sum())
        f0 = min(own, kp1)
        if f0 >= kp1 or f0 % 32 == 0:
            continue
        f1 = f0 + min(32, ring, kp1 - f0)
        cnt += int(f0 // 32 != (f1 - 1) // 32)
    return cnt


# ---- S-bound -----------------------------------------------------------------------------------------------------------
BOUND_RS = (0, 1, 2, 3, 4, 6, 9, 13, 19)
BOUND_K = 5
BOUND_EDGE_NEAR = 0.25            # a power of two: exact products near the origin
BOUND_TOP = 1.0 - 1.0 / 256.0     # a position just below a cell's upper plane, in cells


def directions() -> list:
    return [v for v in np.ndindex(3, 3, 3) if v != (1, 1, 1)]


def _dir(v):
    return np.array(v, np.int64) - 1


def bound_group(base, v, r_p: int, q_frac=None, filler=None, k: int = BOUND_K) -> dict:
    """Points in cell units around the query cell `base`: the query q, k - 1 close points in q's cell, a decoy one cell
    beyond the cube of half-width r_p in direction v (just past its face: the nearest it can be) and a filler inside that
    cube farther than the decoy. q's k nearest are itself, the close points and the decoy, so a search that stopped at
    r_p would keep the filler instead. Returns positions (cells) and the index of q."""
    v = np.asarray(v, np.int64)
    base = np.asarray(base, np.float64)
    f = np.where(v > 0, BOUND_TOP, np.where(v < 0, 0.0, 0.5)) if q_frac is None else np.asarray(q_frac, np.float64)
    q = base + f
    decoy = np.where(v > 0, base + r_p + 1, np.where(v < 0, base - r_p - 1 + BOUND_TOP, q))
    if filler is None:   # the far corner of the cube r_p opposite the decoy
        filler = np.where(v > 0, base - r_p, np.where(v < 0, base + r_p + BOUND_TOP, q))
    away = np.where(v != 0, -np.sign(v), 1).astype(np.float64)
    close = [q + away * (0.02 * (j + 1)) * np.where(v != 0, 1.0, 0.5) for j in range(k - 1)]
    return dict(points=np.vstack([q, close, decoy, filler]), q=0, decoy=k, filler=k + 1)


def _near_cloud(groups, edge=BOUND_EDGE_NEAR) -> np.ndarray:
    return _xyzi(np.vstack([g["points"] for g in groups]) * edge)


def bound_near_cases() -> dict:
    """S-bound (a), near the origin, edge 0.25: for every r_p one cloud of 26 groups along x (one per direction, 3 r_p + 60
    cells apart; the y and z extents are a few cells, so the cubes are clipped there), and six clouds whose query sits
    in its grid's corner cell (the cube clipped on three sides): decoys through the three faces and three edges of the
    positive octant, the filler in the cube's far corner."""
    out = {}
    for r_p in BOUND_RS:
        gap = 3 * r_p + 60
        groups = [bound_group((i * gap, 0, 0), _dir(v), r_p) for i, v in enumerate(directions())]
        pts = _near_cloud(groups)
        off = len(groups[0]["points"])
        out["bound:near:%d" % r_p] = dict(clouds=[pts], mean_k=BOUND_K, cell=BOUND_EDGE_NEAR, r_p=r_p,
                                          queries=[[i * off for i in range(len(groups))]],
                                          decoys=[[i * off + BOUND_K for i in range(len(groups))]])
        clouds, qs, ds = [], [], []
        for v in [(1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (1, 0, 1), (0, 1, 1)]:
            v = np.array(v)
            g = bound_group((0, 0, 0), v, r_p, q_frac=np.where(v > 0, 0.5, 0.25),
                            filler=np.full(3, r_p + BOUND_TOP))
            g["points"] = np.vstack([g["points"][:1], np.maximum(g["points"][1:BOUND_K], 0.01), g["points"][BOUND_K:]])
            clouds.append(_near_cloud([g]))
            qs.append([0])
            ds.append([BOUND_K])
        out["bound:corner:%d" % r_p] = dict(clouds=clouds, mean_k=BOUND_K, cell=BOUND_EDGE_NEAR, r_p=r_p, queries=qs,
                                            decoys=ds)
    return out


def _cell(x, inv) -> int:
    return int(np.floor(F32(F32(x) * F32(inv))))


def _far_group(r_p: int, edge: float, k: int = BOUND_K):
    """S-bound (b): the query in cell 2^19 - 1 (|x * inv| just below 2^19, ulp 2^-5 cell), the decoy in cell 2^19 + r_p
    (ulp 2^-4): its exact product is below that cell's plane but rounds onto it, so it lies less than r_p cells from q
    along x -- inside the bound a kernel with eps = 0 would use. The filler (y offset, cell r_p - 1 on y) has a float
    squared distance between the decoy's and that eps-free bound, so such a kernel stops at r_p with the filler. Returns
    None when this edge gives no such floats."""
    inv = F32(1.0 / edge)
    P = 2 ** 19
    x = F32(P / float(inv))
    while _cell(x, inv) >= P:
        x = np.nextafter(x, F32(-np.inf))
    while _cell(np.nextafter(x, F32(np.inf)), inv) < P:
        x = np.nextafter(x, F32(np.inf))
    xq = x
    x = F32((P + r_p) / float(inv))
    while _cell(x, inv) < P + r_p:
        x = np.nextafter(x, F32(np.inf))
    while _cell(np.nextafter(x, F32(-np.inf)), inv) >= P + r_p:
        x = np.nextafter(x, F32(-np.inf))
    xp = x
    dx = F32(xp - xq)
    d_decoy = float(F32(dx * dx))
    cell = 1.0 / float(inv)
    b0 = bound_at(r_p, 0.0, cell)
    if not d_decoy < b0:
        return None
    y = F32(math.sqrt(b0))
    while float(F32(y * y)) > b0:
        y = np.nextafter(y, F32(-np.inf))
    if not float(F32(y * y)) > d_decoy or _cell(y, inv) > r_p:
        return None
    pts = [(xq, 0, 0)] + [(xq, F32(0.05 * cell * (j + 1)), 0) for j in range(k - 1)] + [(xp, 0, 0), (xq, y, 0)]
    return _xyzi(pts)


FAR_EDGES = tuple(0.3 + 0.0007 * i for i in range(200))


def bound_far_cases() -> dict:
    out = {}
    for r_p in BOUND_RS[1:]:
        for edge in FAR_EDGES:
            c = _far_group(r_p, edge)
            if c is not None:
                out["bound:far:%d" % r_p] = dict(clouds=[c], mean_k=BOUND_K, cell=edge, r_p=r_p, queries=[[0]],
                                                 decoys=[[BOUND_K]], far=True)
                break
        else:
            raise AssertionError("no edge gives a far bound case for r = %d" % r_p)
    return out


def built_stop(case, plan, c: int, qi: int) -> int:
    """the half-width the search of query qi of cloud c must stop at: the first growth step past r_p whose bound reaches
    the query's k-th value (taken from the exact neighbours), or whose cube covers the grid."""
    x = np.asarray(case["clouds"][c], F32)
    kth = float(sor_np.knn_sq(np.ascontiguousarray(x[:, :3]), case["mean_k"] + 1)[qi, -1])
    g = plan["grids"][c]
    cq = cells_of(x[qi:qi + 1], plan["inv"])[0] - g["min_b"]
    eps = search_eps(g)
    r = next_r(case["r_p"])
    while not (bound_at(r, eps, plan["cell"]) >= kth or ((cq - r <= 0) & (cq + r >= g["div"] - 1)).all()):
        r = next_r(r)
    return r


# ---- S-plan ------------------------------------------------------------------------------------------------------------
def cluster(centre, n: int = 27, step: float = 0.3) -> np.ndarray:
    """n points on a small lattice of `step` (in the units of centre) around it."""
    s = int(round(n ** (1 / 3)))
    g = (np.arange(s) - (s - 1) / 2.0) * step
    a, b, c = np.meshgrid(g, g, g, indexing="ij")
    return np.column_stack([a.ravel(), b.ravel(), c.ravel()])[:n] + np.asarray(centre, np.float64)


def two_corners(div, edge: float = 1.0) -> np.ndarray:
    """two clusters well inside the first and last cell of a grid of div cells (forced edge `edge`, a power of two)."""
    d = np.asarray(div, np.float64)
    a = cluster((0.5, 0.5, 0.5), step=0.2)
    b = cluster(d - 0.5, step=0.2)
    return _xyzi(np.vstack([a, b]) * edge)


PASS_DIVS = {1: (16, 16, 1), 2: (256, 256, 1), 3: (256, 256, 256), 4: (2048, 2048, 1024), 5: (2048, 2048, 1025),
             6: (65536, 65536, 4096), 7: (131072, 131072, 131072)}


def plan_cases() -> dict:
    out = {}
    for p, div in PASS_DIVS.items():   # idx bits 8, 16, 24, 32, 33, 44, 51
        out["plan:passes:%d" % p] = dict(clouds=[two_corners(div)], mean_k=5, cell=1.0, passes=p)
    # 8 passes: the floor through extent (a forced edge far below it): 2^19 / (1 + 2^-10) cells on every axis, 57 bits
    L = 1000.0
    out["plan:passes:8"] = dict(clouds=[_xyzi(np.vstack([cluster((0, 0, 0), step=5e-4), cluster((L, L, L), step=5e-4)]))],
                                mean_k=5, cell=1e-9, passes=8, floor="extent")
    # the floor through magnitude: a dense patch at UTM-sized coordinates, other extents small
    utm = cluster((5.0e5, 4.2e6, 30.0), n=64, step=0.5)
    out["plan:floor:utm"] = dict(clouds=[_xyzi(utm)], mean_k=10, cell=1e-3, floor="magnitude")
    # 16 clouds, 12 index bits: frame bits 4 (16 bits, 2 passes) or 5 with a non-finite row (17 bits, 3 passes)
    sixteen = [two_corners((64, 64, 1)) + np.array([k * 1000.0, 0, 0, 0], F32) for k in range(16)]
    out["plan:frames:16"] = dict(clouds=sixteen, mean_k=5, cell=1.0)
    bad = [c.copy() for c in sixteen]
    bad[7] = np.concatenate([bad[7], np.array([[np.nan, 0, 0, 0]], F32)])
    out["plan:frames:16+sentinel"] = dict(clouds=bad, mean_k=5, cell=1.0)
    # the table limit: n_clouds << idx_bits == 2^25 (table) and one bit over (binary searches)
    out["plan:table:1x25"] = dict(clouds=[two_corners((1 << 13, 1 << 12, 1))], mean_k=5, cell=1.0)
    out["plan:table:1x26"] = dict(clouds=[two_corners((1 << 13, 1 << 13, 1))], mean_k=5, cell=1.0)
    out["plan:table:16x21"] = dict(clouds=[two_corners((1 << 11, 1 << 10, 1)) for _ in range(16)], mean_k=5, cell=1.0)
    out["plan:table:16x22"] = dict(clouds=[two_corners((1 << 11, 1 << 11, 1)) for _ in range(16)], mean_k=5, cell=1.0)
    # the clamps: extents near +-FLT_MAX (the estimate exceeds 1e36) and a cloud a few 1e-31 across (below 1e-30)
    big = np.float32(3.0e38)
    huge = np.vstack([cluster((0, 0, 0), n=27, step=0.1), [[big, 0, 0], [-big, 0, 0], [0, big, -big], [big, big, big]]])
    out["plan:clamp:max"] = dict(clouds=[_xyzi(huge)], mean_k=3, clamp="max")
    tiny = cluster((0, 0, 0), n=27, step=1e-31)
    sub = np.vstack([tiny, np.array([[1e-40, 2e-40, 0], [3e-44, 0, -1e-39]])])
    out["plan:clamp:min"] = dict(clouds=[_xyzi(sub)], mean_k=3, clamp="min")
    return out


# ---- S-sums ------------------------------------------------------------------------------------------------------------
P1_M = 14529495                   # odd, and fl(m * m) = 3 * 2^46: its float square has its lowest set bit 46 above 2 e_min


def pairs_cloud(seps, spacing: float, small_last=()) -> np.ndarray:
    """isolated pairs along x, one per separation, on a 3-D grid of `spacing`, then the pairs of small_last at the
    origin side, last in index order. With mean_k = 1 each point's distance is its pair's separation exactly when the
    separation is m * 2^e with m < 2^12 (the square, its root and the mean are exact)."""
    seps = list(seps)
    n = len(seps)
    s = max(1, int(math.ceil(n ** (1 / 3))))
    pts = []
    for i, d in enumerate(seps):
        a, b, c = i % s + 1, (i // s) % s, i // (s * s)
        o = np.array([a * spacing, b * spacing, c * spacing])
        pts += [o, o + np.array([d, 0.0, 0.0])]
    for j, d in enumerate(small_last):
        o = np.array([0.0, 0.0, j * spacing])
        pts += [o, o + np.array([d, 0.0, 0.0])]
    x = np.array(pts, np.float64)
    c = _xyzi(x)
    assert (c[:, :3].astype(np.float64) == x).all(), "pair coordinates must be exact floats"
    return c


def sums_cases() -> dict:
    out = {}
    # the sum of 2^53 +- : 4095 / 4096 pairs at 2^40 and a pair at 1.0 (values 2^40 x 8190 + 1 + 1 = 2^53 - 2^41 + 2; with
    # 4096 pairs 2^53 + 2); the squares fail either way
    out["sums:2p40:4095"] = dict(clouds=[pairs_cloud([2.0 ** 40] * 4095, 2.0 ** 42, [1.0])], mean_k=1, path=2)
    out["sums:2p40:4096"] = dict(clouds=[pairs_cloud([2.0 ** 40] * 4096, 2.0 ** 42, [1.0])], mean_k=1, path=3, tight=1)
    # the square sum alone: values 2^-20 (square 2^-40) and 2^6 (square 2^12): 2 * 2^52 + 2 units of 2^-40 -> over;
    # (2^12 - 1) * 2^-8 -> 2^53 - 2^42 + 2 -> under
    u = 2.0 ** -20
    out["sums:sq:over"] = dict(clouds=[pairs_cloud([2.0 ** 26 * u], 4.0 * 2 ** 6, [u])], mean_k=1, path=2, tight=2)
    out["sums:sq:under"] = dict(clouds=[pairs_cloud([(2 ** 12 - 1) * 2.0 ** 14 * u], 4.0 * 2 ** 6, [u])], mean_k=1,
                                path=0)
    # both: values 2^-30 and 2^52 * 2^-30 (sum 2^53 + 2 units) -> 3; 2^51 units -> sum under, squares over -> 2
    u = 2.0 ** -30
    out["sums:both:over"] = dict(clouds=[pairs_cloud([2.0 ** 52 * u], 2.0 ** 25, [u])], mean_k=1, path=3, tight=1)
    out["sums:both:under"] = dict(clouds=[pairs_cloud([2.0 ** 51 * u], 2.0 ** 25, [u])], mean_k=1, path=2)
    # the sum alone: its smallest value m * 2^-23 has a float square whose lowest set bit is 2^46 units above 2 e_min, so
    # the squares pass while 256 values of 2^45 units reach 2^53 units (254 stay below)
    u = 2.0 ** -23
    vj = P1_M * u
    out["sums:sum:over"] = dict(clouds=[pairs_cloud([2.0 ** 45 * u] * 128, 2.0 ** 24, [vj])], mean_k=1, path=1, tight=1)
    out["sums:sum:under"] = dict(clouds=[pairs_cloud([2.0 ** 45 * u] * 127, 2.0 ** 24, [vj])], mean_k=1, path=0)
    # subnormal squares: separations 2^-70, 3 * 2^-71, 2^-74 (squares 2^-140 ... 2^-148), alone (exact: path 0) and with a
    # pair at 1.0 (e_min -74: both serial)
    tinies = [2.0 ** -70, 3.0 * 2.0 ** -71, 2.0 ** -74, 5.0 * 2.0 ** -73]
    out["sums:subnormal"] = dict(clouds=[pairs_cloud(tinies, 2.0 ** -60)], mean_k=1, path=0)
    out["sums:subnormal+1"] = dict(clouds=[pairs_cloud([1.0], 8.0, tinies)], mean_k=1, path=3)
    # overflow: separations 2^64 (square inf: the distance is inf) next to 2^63 (square 2^126) and 1.0
    out["sums:overflow"] = dict(clouds=[pairs_cloud([2.0 ** 63, 2.0 ** 64, 1.0], 2.0 ** 66)], mean_k=1, path=3)
    out["sums:n_valid=2"] = dict(clouds=[pairs_cloud([0.75], 4.0)], mean_k=1, path=0)
    # strides of the parallel pass and of the serial tiles: both paths (the serial chain forced too), small values last
    for n in (1023, 1024, 1025, 4095, 4097, 9000):
        rng = np.random.default_rng(n)
        c = _xyzi(rng.normal(scale=[20.0, 20.0, 2.0], size=(n, 3)))
        out["sums:size:%d" % n] = dict(clouds=[c], mean_k=3, serial_too=True)
    # 16 clouds on different paths in one call
    keys = ["sums:sq:over", "sums:sq:under", "sums:both:over", "sums:both:under", "sums:sum:over", "sums:sum:under",
            "sums:subnormal", "sums:subnormal+1", "sums:overflow", "sums:n_valid=2"]
    clouds = [out[k]["clouds"][0] for k in keys]
    clouds += [pairs_cloud([0.5, 0.25, 0.125], 8.0), np.zeros((0, 4), F32), pairs_cloud([3.0], 16.0, [2.0 ** -40]),
               pairs_cloud([2.0 ** 30] * 3, 2.0 ** 33, [2.0 ** -23]), pairs_cloud([1.5] * 7, 8.0),
               np.full((3, 4), np.nan, F32)]
    out["sums:16-clouds"] = dict(clouds=clouds, mean_k=1)
    return out


# ---- S-select ----------------------------------------------------------------------------------------------------------
def select_cases() -> dict:
    """distances {1, 1, 2, 2, 3, 3}: mean exactly 2, so std_mul 0 puts two distances on the threshold (kept; removed when
    negative). Empty clouds first, in the middle and last of a multi call."""
    six = pairs_cloud([1.0, 2.0, 3.0], 16.0)
    e = np.zeros((0, 4), F32)
    return {"select:on-threshold": dict(clouds=[six], mean_k=1, std_mul=0.0, negative_too=True),
            "select:empties": dict(clouds=[e, six, e, pairs_cloud([0.5, 4.0, 1.0, 1.0], 32.0), e], mean_k=1,
                                   std_mul=0.0, negative_too=True)}


def slot_cases() -> dict:
    out = {}
    for k in SLOT_MEAN_KS:
        out["slots:lattice:%d" % k] = dict(clouds=[slot_lattice(k)], mean_k=k, sqrt_modes=(0, 1))
        out["slots:blob:%d" % k] = dict(clouds=[slot_blob(k)], mean_k=k, sqrt_modes=(0, 1))
    for k in SLOT_EXACT_KS:
        out["slots:exact:%d" % k] = dict(clouds=[slot_exact(k)], mean_k=k, sqrt_modes=(0, 1))
    for k in (40, 62, 126):
        out["slots:cells:%d" % k] = dict(clouds=[slot_cells(k)], mean_k=k, cell=SLOT_CELL, sqrt_modes=(0, 1))
    return out


def sor_cases() -> dict:
    out = {}
    for part in (slot_cases(), bound_near_cases(), bound_far_cases(), plan_cases(), sums_cases(), select_cases()):
        out.update(part)
    return out


# ---- the cost cliff of one edge for every cloud of a call -----------------------------------------------------------------
def cliff_clouds(seed: int = 0) -> list:
    """a dense cloud (1 M points in a 2 m x 2 m patch) and a sparse one (200 points in a 1 km cube) in one call: the edge
    comes from the dense cloud (3.7 mm), and the sparse cloud's searches then cross ~10^5 cells. NOT for the GPU."""
    rng = np.random.default_rng(seed)
    dense = _xyzi(np.column_stack([rng.uniform(0, 2, (1_000_000, 2)), np.zeros(1_000_000)]))
    sparse = _xyzi(rng.uniform(0, 1000, (200, 3)))
    return [dense, sparse]
