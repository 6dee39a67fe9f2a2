"""The edge-case generators (tests/edge_inputs.py) on the CPU: their inputs reach the fragile spots they are meant to reach,
and the two CPU references -- the C++ oracle and the numpy restatement -- agree on every one of them."""
import os
import re

import numpy as np
import pytest

import edge_inputs as E
from helpers import cloud_dict, host_function
from oracle import np_oracle

F32 = np.float32


@pytest.mark.parametrize("leaf", E.LEAVES)
def test_lattice_points_discriminate_the_cell_formula(leaf):
    """A kernel that computed x / leaf, or rounded the product x * inv towards zero, must misplace some lattice points: at
    least 2 % of their coordinates fall into another cell under either formula. Power-of-two leaves have exact products --
    no formula can differ there -- and their planes k * leaf are exact, so x0 lies on the plane and x0 - 1 ulp below it."""
    x = E.lattice_cloud(11, leaf)[:, :3]
    d = E.lattice_discrimination(leaf, x)
    if float(np.log2(leaf)).is_integer():
        assert d["either"] == 0.0
        v = E.lattice_values(leaf, np.arange(-5, 6))
        x0, below = v[:11], v[11 * 2:11 * 3]     # x0, then +1 ulp, then -1 ulp
        assert (np.floor(x0 * E.inv_of(leaf)) == np.arange(-5, 6)).all()
        assert (np.floor(below * E.inv_of(leaf)) == np.arange(-5, 6) - 1).all()
    else:
        assert d["vs_division"] >= 0.02 and d["vs_round_to_zero"] >= 0.015, d
    assert (x < 0).any() and (x > 0).any() and (x == 0).any()


def test_box_limit_points_land_on_the_limits():
    """Family B: after the unfused transform the box limits, and one ulp either side of each, occur in the data."""
    t = (1.25, 0.5, 0.375)
    box = [(-2.5, 7.25), (-3.0, 3.5), (-1.5, 2.0)]
    x = E.box_limit_cloud(5, t, box, intensity_window=(10.0, 200.0))
    y = np_oracle.transform(x, E.identity_extrinsic(t)[:3].reshape(-1))
    for a in range(3):
        for v in E.limit_values(*box[a]):
            assert (y[:, a] == v).sum() >= 3, (a, v)
    for v in E.limit_values(10.0, 200.0):
        assert (y[:, 3] == v).sum() >= 3


def test_signed_zero_and_subnormals_survive_the_transform():
    x = E.signed_zero_subnormal_cloud(3)
    y = np_oracle.transform(x, E.identity_extrinsic((-0.0, -0.0, -0.0)).reshape(-1))
    special = (np.abs(x[:, :3]) < np.finfo(F32).tiny).any(axis=1) | (np.abs(x[:, 3]) < np.finfo(F32).tiny)
    assert (y[special].view(np.uint32) == x[special].view(np.uint32)).all(), "-0.0 and subnormals must keep every bit"
    sub = (np.abs(y[:, :3]) > 0) & (np.abs(y[:, :3]) < np.finfo(F32).tiny)
    assert sub.any(axis=0).all() and (np.signbit(y[:, :3]) & (y[:, :3] == 0)).any(axis=0).all()


@pytest.mark.parametrize("div,overflow,bits", [(E.DIV_2P31, True, 31), (E.DIV_2P31_PLUS, True, 32), (E.DIV_2P32, True, 32),
                                               (E.DIV_2P32_PLUS, True, 33), (E.DIV_GUARD_BELOW, False, 31),
                                               (E.DIV_GUARD_ABOVE, True, 32)])
def test_grid_cloud_has_the_intended_grid(oracle, div, overflow, bits):
    x = E.grid_cloud(1, div, n_filler=2000)
    o = oracle.voxelgrid(x, [1.0] * 3, 1, True, force64=True)
    assert o["div_b"].tolist() == list(div) and o["pcl_overflow"] == overflow
    assert E.bits_for(int(np.prod(np.asarray(div, np.int64)))) == bits


def test_guard_and_key_grid_disagree(oracle):
    """Points at 0.9 and a - 0.9: PCL's d is a - 1 per axis, the key grid a cells. At a = 1291 the guard passes
    (1290^3 <= INT32_MAX) while the grid holds more than INT32_MAX cells."""
    x = E.grid_cloud(2, E.DIV_GUARD_ABOVE, n_filler=2000, inset=0.9)
    o = oracle.voxelgrid(x, [1.0] * 3, 1, True, force64=True)
    assert o["div_b"].tolist() == list(E.DIV_GUARD_ABOVE) and not o["pcl_overflow"]
    assert int(np.prod(o["div_b"].astype(np.int64))) > 2**31 - 1


# ---- the two references on every family --------------------------------------------------------------------------------
def edge_cases():
    """(name, clouds [(xyzi, m, is_dense)], passes, leaf) -- the frames the GPU edge tests run, small enough for the CPU."""
    cases = []
    for leaf in E.LEAVES:
        x = E.lattice_cloud(100, leaf, n_lattice=6000, n_filler=3000)
        cases.append(("A-leaf%g" % leaf, [(x, E.identity_extrinsic((0, 0, 0)), 1)], [], leaf))
    t = (1.25, 0.5, 0.375)
    box = [(-2.5, 7.25), (-3.0, 3.5), (-1.5, 2.0)]
    for dense in (1, 0):
        x = E.box_limit_cloud(7, t, box, intensity_window=(10.0, 200.0))
        if not dense:
            x[::97, 1] = np.nan
        passes = [(a, box[a][0], box[a][1], 0) for a in range(3)]
        cases.append(("B-box-dense%d" % dense, [(x, E.identity_extrinsic(t), dense)], passes, 0.25))
        cases.append(("B-box-int-dense%d" % dense, [(x, E.identity_extrinsic(t), dense)], passes + [(3, 10.0, 200.0, 0)], 0.1))
    m = E.rotated_extrinsic(0.7, (3.0, -2.0, 1.5), pitch=0.05)
    x = E.lattice_cloud(8, 0.1, n_lattice=4000, n_filler=4000)
    lim = E.limits_from_data(np_oracle.transform(x, m.reshape(-1)))
    cases.append(("B-rotated", [(x, m, 1)], [(a, lo, hi, 0) for a, lo, hi in lim], 0.1))
    z = E.signed_zero_subnormal_cloud(9)
    mz = E.identity_extrinsic((-0.0, -0.0, -0.0))
    for lo, hi in ((0.0, 0.5), (-0.5, 0.0)):
        cases.append(("B-zero-%g-%g" % (lo, hi), [(z, mz, 1)], [(a, lo if a == 0 else -1.0, hi if a == 0 else 1.0, 0)
                                                                  for a in range(3)] + [(3, 0.0, 255.0, 0)], 0.05))
    for leaf in (0.02, 0.05, 0.1):
        x = E.offset_cloud(20, leaf, n=12000)
        cases.append(("C-map-leaf%g" % leaf, [(x, E.identity_extrinsic((0, 0, 0)), 1)], [], leaf))
    xs = E.lattice_cloud(21, 0.05, n_lattice=5000, n_filler=5000)
    mk = E.rotated_extrinsic(-1.1, (2500.0, -3800.0, 35.0))
    cases.append(("C-km-extrinsic", [(xs, mk, 1)], [(2, 30.0, 40.0, 0)], 0.05))
    for div in (E.DIV_2P31, E.DIV_2P31_PLUS, E.DIV_GUARD_BELOW, E.DIV_GUARD_ABOVE):
        cases.append(("D-%s" % "x".join(map(str, div)), [(E.grid_cloud(3, div, n_filler=4000), E.identity_extrinsic((0, 0, 0)), 1)],
                      [], 1.0))
    cases.append(("D-guard-disagrees", [(E.grid_cloud(4, E.DIV_GUARD_ABOVE, n_filler=4000, inset=0.9),
                                         E.identity_extrinsic((0, 0, 0)), 1)], [], 1.0))
    return cases


CASES = edge_cases()


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("min_points", [1, 2])
def test_oracles_agree_on_edge_inputs(oracle, case, min_points):
    name, clouds, passes, leaf = case
    cds = [cloud_dict(x, m, dense) for x, m, dense in clouds]
    c = oracle.merge_frame(cds, passes, [leaf] * 3, min_points, True, True)
    n = np_oracle.merge_frame(cds, passes, [leaf] * 3, min_points, True, True)
    assert c["n_survivors"] == len(n["survivor_src"]) > 0
    assert (c["survivor_src"] == n["survivor_src"]).all()
    assert (c["survivor_xyzi"].view(np.uint32) == n["survivor_xyzi"].view(np.uint32)).all()
    v = n["voxel"]
    assert c["min_b"].tolist() == v["min_b"].tolist() and c["div_b"].tolist() == v["div_b"].tolist()
    assert c["pcl_overflow"] == v["pcl_overflow"]
    assert (c["point_idx"] == v["point_idx"]).all(), "voxel membership"
    assert (c["idx"] == v["idx"]).all() and (c["count"] == v["count"]).all()
    np.testing.assert_allclose(c["centroid_f64"], v["centroid_f64"], rtol=1e-12, atol=1e-12)
    assert c["n_voxels"] > 0


# ---- R: run layouts of the centroid pass ---------------------------------------------------------------------------------
VOXEL_CU = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "cloud_merger_b200", "csrc", "cm_voxel.cu")


def test_mirrored_centroid_constants_match_the_source():
    """The layouts aim at k_voxel_centroid's tiles, threads, hand-over point and tail rounds through constants mirrored in
    edge_inputs.py: a retune of the kernel must fail here, not quietly move the edges away from the layouts."""
    src = open(VOXEL_CU).read()

    def const(name):
        m = re.search(r"constexpr\s+\w+\s+%s\s*=\s*([^;]+);" % name, src)
        assert m, name
        return m.group(1).strip()

    def define(name):
        m = re.search(r"#define\s+%s\s+(.+?)\s*(?://.*)?$" % name, src, re.M)
        assert m, name
        return m.group(1).strip()
    assert int(const("VX_THREADS")) == E.VX_THREADS
    assert int(const("CE_IPT")) == E.CE_IPT
    assert const("CE_TILE") == "VX_THREADS * CE_IPT" and E.CE_TILE == E.VX_THREADS * E.CE_IPT == 2048
    assert int(const("CE_TAIL_INLINE").rstrip("u")) == E.CE_TAIL_INLINE
    assert int(const("CE_TAIL_U")) == E.CE_TAIL_U
    assert const("CE_TAIL_ITEMS") == "CE_TAIL_U * VX_THREADS" and E.CE_TAIL_ITEMS == E.CE_TAIL_U * E.VX_THREADS
    assert int(const("CE_SEG_SMEM_FRAMES").rstrip("u")) == E.CE_SEG_SMEM_FRAMES
    assert int(define("CE_ASYNC_GATHER")) == 1
    assert define("CE_MIN_CTAS") == "(CE_ASYNC_GATHER ? %d : 4)" % E.CE_MIN_CTAS
    assert "std::min<uint32_t>(tiles, %du * (uint32_t)CE_MIN_CTAS)" % E.B200_SMS in src
    # the persistent grid holds fewer tiles than R-persist has: every CTA takes several and alternates its point buffers
    runs, _ = E.layout("persist")
    assert sum(runs) / E.CE_TILE > 3 * E.B200_SMS * E.CE_MIN_CTAS


def _runs_of(x, min_points=1):
    """From the numpy oracle alone: the finite rows in sorted order (stable: ascending row index inside a voxel), their voxel
    indices, and the sorted positions where runs start."""
    o = np_oracle.voxelgrid(x, [1.0] * 3, min_points, True, True)
    pidx = o["point_idx"]
    fin = np.nonzero(pidx >= 0)[0]
    order = fin[np.argsort(pidx[fin], kind="stable")]
    keys = pidx[order]
    starts = np.nonzero(np.r_[True, keys[1:] != keys[:-1]])[0] if len(keys) else np.zeros(0, np.int64)
    return order, keys, starts, o


def _check_marks(name, runs, marks, starts, m_items):
    w = E.centroid_walk(starts, m_items)
    at = {int(s): i for i, s in enumerate(starts)}
    bounds = set(int(s) for s in starts) | {m_items}

    def run_at(s, e):
        assert s in at and e in bounds and (at[s] + 1 == len(starts) or int(starts[at[s] + 1]) == e), (name, s, e)
        return at[s]
    for e in marks.get("bounds", []):
        for d in E.R_BOUND_OFFSETS:
            assert e + d in bounds, (name, e, d)
    if "leave" in marks:
        idx = [run_at(s, e) for s, e in marks["leave"]]
        reps = len(idx) // len(E.LEAVE_PAST + E.LEAVE_ROUND)   # R-persist repeats the block
        assert reps and sorted(int(w["past"][i]) for i in idx) == sorted((E.LEAVE_PAST + E.LEAVE_ROUND) * reps)
        inline = [i for i in idx if 0 < w["past"][i] <= E.CE_TAIL_INLINE]
        handed = [i for i in idx if w["handed"][i]]
        assert any(w["past"][i] == E.CE_TAIL_INLINE for i in inline), "a run that fills the inline walk exactly"
        assert any(w["past"][i] == E.CE_TAIL_INLINE + 1 for i in handed), "a run handed over at its 25th point past the tile"
        tails = w["tail_items"][handed]
        for d in (-1, 0, 1):   # tail rounds that end one short of, on and one past a round boundary
            for k in (1, 2, 3):
                assert (tails == k * E.CE_TAIL_ITEMS + d).any(), (k, d)
        assert {(-s) % E.CE_TILE or E.CE_TILE for s, _ in marks["leave"]} == set(E.LEAVE_BACK)   # where the heads sit
    for s, e in marks.get("whole", []):
        i = run_at(s, e)
        assert s % E.CE_TILE == 0 and (e - s) % E.CE_TILE == 0
        k = (e - s) // E.CE_TILE
        assert w["past"][i] == (k - 1) * E.CE_TILE   # the k - 1 tiles after the first have no head: they publish 0 voxels
    if "dense-last" in marks:
        per_tile = np.bincount(w["tile"])
        assert (per_tile == E.CE_TILE).any() and (per_tile == 256).any() and (per_tile == 257).any()
        for s, e in marks["dense-last"]:
            i = run_at(s, e)
            assert w["handed"][i] and per_tile[w["tile"][i]] > 256
            assert i + 1 == len(starts) or w["tile"][i + 1] != w["tile"][i], "the handed-over run is its tile's last"
    if name.startswith("end:"):
        assert m_items == sum(runs)
        kind = name[4:]
        if kind in ("2T-1", "2T", "2T+1"):
            assert m_items == 2 * E.CE_TILE + {"2T-1": -1, "2T": 0, "2T+1": 1}[kind]
        if kind == "M7":
            assert m_items < E.CE_IPT
        if kind.startswith("handover"):
            (s, e), = marks["end"]
            i = run_at(s, e)
            assert e == m_items and w["handed"][i]
            if kind == "handover-round":
                assert w["tail_items"][i] == E.CE_TAIL_ITEMS   # the second round starts at M: only the limit ends it
            else:
                assert m_items % E.CE_TILE and w["tile"][i] + 1 == m_items // E.CE_TILE
    if name.startswith("minpts:"):
        m, last = (int(v) for v in name.split(":")[1:])
        crossed = set()
        for s, e in marks["straddle"]:
            run_at(s, e)
            ahead = s + m - 1                      # the item the min-points test of the head looks at
            for step in (E.CE_IPT, E.VX_THREADS, E.CE_TILE):
                if ahead // step != s // step:
                    crossed.add(step)
        assert crossed == {E.CE_IPT, E.VX_THREADS, E.CE_TILE}
        (s, e), = marks["end"]
        assert e == m_items and e - s == last and ((s + m - 1 >= m_items) == (last < m))


@pytest.mark.parametrize("name", E.R_LAYOUTS + E.R_MINPTS + ("persist",))
def test_run_layout_positions(name):
    """The oracle's own runs of every R layout (recomputed from its keys and its stable order) are exactly the intended
    ones, and they sit where the layout aims: R-bounds offsets, the inline walk and the hand-over at the 25th point, tail
    rounds ending one short of, on and one past a round, whole tiles without a head, dense tiles, the end of the cloud, the
    min-points look-ahead across thread, warp and tile edges and past M."""
    runs, marks = E.layout(name, seed=7)
    x = E.run_layout_cloud(runs, seed=len(name))
    order, keys, starts, _ = _runs_of(x)
    assert np.diff(np.r_[starts, len(keys)]).tolist() == list(runs)
    assert (keys[starts] == np.arange(len(runs))).all(), "run r is cell r"
    assert len(order) < 8 or not (order[1:] > order[:-1]).all(), "the gather must be scattered"
    _check_marks(name, runs, marks, starts, len(keys))


@pytest.mark.parametrize("name", ["seg3", "seg300"])
def test_batch_layout_positions(name):
    """The frame-split layouts: every frame's runs are the intended ones; seg3 puts voxel index 0 on both sides of a frame
    edge inside an inline walk and inside a tail round, and has handed-over runs in a tile that straddles frames and in one
    that does not; seg300 has more frames than are staged in shared memory, empty frames, and frame edges at every R-bounds
    offset."""
    runs, cuts, marks = E.batch_layout(name, seed=3)
    frames = E.split_runs(runs, cuts)
    clouds = E.run_layout_frames(runs, cuts, seed=11)
    fs = np.r_[0, cuts]
    assert len(frames) == len(cuts) + 1 and np.diff(np.r_[fs, sum(runs)]).tolist() == [len(c) for c in clouds]
    first_last = []
    for f, (fr, x) in enumerate(zip(frames, clouds)):
        if not fr:
            first_last.append(None)
            continue
        _, keys, starts, _ = _runs_of(x)
        assert np.diff(np.r_[starts, len(keys)]).tolist() == fr, f
        first_last.append((int(keys[0]), int(keys[-1])))
    # the kernel's view: runs of equal (frame, index) over the concatenated frames
    starts = np.unique(np.r_[fs, np.cumsum(runs)[:-1]])
    starts = starts[starts < sum(runs)]
    w = E.centroid_walk(starts, sum(runs), fs)
    assert (w["handed"] & w["straddles"]).any() and (w["handed"] & ~w["straddles"]).any()
    same = [(f, c) for f, c in enumerate(cuts) if first_last[f] and first_last[f + 1] and first_last[f][1] == first_last[f + 1][0]]
    kinds = set()
    for f, c in same:
        i = int(np.searchsorted(starts, c)) - 1          # the run that ends at the frame edge
        edge = min((int(w["tile"][i]) + 1) * E.CE_TILE, sum(runs))
        if w["start"][i] < edge < c:
            kinds.add("tail" if c - edge > E.CE_TAIL_INLINE else "inline")
    assert kinds == {"inline", "tail"}, kinds
    if name == "seg300":
        assert len(frames) == 300 > E.CE_SEG_SMEM_FRAMES and sum(1 for f in frames if not f) >= 3
        for e in marks["bounds"]:
            for d in E.R_BOUND_OFFSETS:
                assert e + d in cuts


def _seq_sum(p):
    return np.cumsum(np.asarray(p, F32), axis=0, dtype=F32)[-1] if len(p) else np.zeros(4, F32)


@pytest.mark.parametrize("name", ["bounds", "leave", "dense", "end:handover-round", "end:handover-partial",
                                  "minpts:1025:1024", "persist"])
def test_run_layout_sums_see_every_point_and_their_order(name):
    """Every run that leaves its tile, and every run at an R-bounds edge, has a float32 sequential sum (ascending row order,
    as the kernel and the float oracle add) that differs bitwise from the same sum without the point at the tile edge, with
    that point counted twice, and -- from 3 points on -- from the reversed sum: a kernel that drops, repeats or re-orders a
    point there cannot match the oracle bit for bit."""
    runs, marks = E.layout(name, seed=7)
    x = E.run_layout_cloud(runs, seed=len(name))
    order, keys, starts, _ = _runs_of(x)
    m_items = len(keys)
    w = E.centroid_walk(starts, m_items)
    ends = w["end"]
    target = set(np.nonzero(w["past"] > 0)[0].tolist())
    for e in marks.get("bounds", []):
        target |= set((np.searchsorted(starts, [e + d for d in E.R_BOUND_OFFSETS], side="right") - 1).tolist())
    assert target
    reversed_checked = 0
    for i in sorted(target):
        s, e = int(starts[i]), int(ends[i])
        pts = x[order[s:e]]
        edge = min(max((s // E.CE_TILE + 1) * E.CE_TILE, s), e - 1) - s   # the first point past the tile, else the last
        ref = _seq_sum(pts)
        drop = _seq_sum(np.delete(pts, edge, axis=0))
        dup = _seq_sum(np.insert(pts, edge, pts[edge], axis=0))
        assert (ref.view(np.uint32) != drop.view(np.uint32)).any(), (name, s, e, "drop")
        assert (ref.view(np.uint32) != dup.view(np.uint32)).any(), (name, s, e, "twice")
        if e - s >= 3:   # (a + b == b + a)
            assert (ref.view(np.uint32) != _seq_sum(pts[::-1]).view(np.uint32)).any(), (name, s, e, "reversed")
            reversed_checked += 1
    assert reversed_checked


R_ORACLE_CASES = [(n, 1, 0, False) for n in E.R_LAYOUTS] + [(n, int(n.split(":")[1]), 0, False) for n in E.R_MINPTS] + \
    [("leave", 2, 0, True), ("bounds", 3, 0, True), ("leave", 1, 5000, False), ("dense", 2, 300, True), ("persist", 2, 0, False)]


@pytest.mark.parametrize("case", R_ORACLE_CASES, ids=["%s-mp%d-nf%d-far%d" % c for c in R_ORACLE_CASES])
def test_oracles_agree_on_run_layouts(oracle, case):
    """The C++ oracle and the numpy restatement agree on every R layout (with non-finite rows and far corners too): the
    number of voxels, their indices and counts, and the membership of every point."""
    name, min_points, n_nf, far = case
    runs, _ = E.layout(name, seed=7)
    x = E.run_layout_cloud(runs, seed=len(name), n_nonfinite=n_nf, far=far)
    c = oracle.voxelgrid(x, [1.0] * 3, min_points, True, force64=True, is_dense=n_nf == 0)
    n = np_oracle.voxelgrid(x, [1.0] * 3, min_points, True, True)
    assert c["n"] == len(n["idx"]) and (c["idx"] == n["idx"]).all() and (c["count"] == n["count"]).all()
    assert (c["point_idx"] == n["point_idx"]).all()
    np.testing.assert_allclose(c["centroid_f64"], n["centroid_f64"], rtol=1e-12, atol=1e-12)
    if far:
        assert E.bits_for(int(np.prod(c["div_b"].astype(np.int64)))) == 33
    else:
        assert c["min_b"].tolist() == [0, 0, 0] and c["n"] == sum(1 for r in runs if r >= min_points)


# ---- N: radius outlier removal ------------------------------------------------------------------------------------------
def _src(name):
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "cloud_merger_b200", "csrc", name)) as f:
        return f.read()


def test_ror_constants_match_the_source():
    """The N-family restatement mirrors the kernels' constants; a retune must fail here rather than miss the edges."""
    ror, vox = _src("cm_outlier.cu"), _src("cm_voxel.cu")
    run, front, keys, table = (host_function(f) for f in ("radius_outlier_run", "cell_keys_begin", "cell_keys_sort",
                                                          "enqueue_cell_table"))
    assert "(float)radius * 1.00390625f" in run and E.ROR_MARGIN == 1.00390625
    assert "worst >= (1 << 14)" in ror and E.ROR_BOUND == 1 << 14
    assert "w.plan_idx_bits <= 25 && ((uint64_t)n_clouds << w.plan_idx_bits) <= (1ull << 25)" in table and E.ROR_TABLE_LOG2 == 25
    assert 'enqueue_cell_table(h, vp, "CM_ROR_NO_TABLE", rp, st)' in run
    # the launches cm_launch_count reports for the call (ror_launches): a bounding box per cloud and the table in the shared
    # front end, the count in the run
    assert front.count("++w.launches;") == 1 and table.count("++w.launches;") == 1 and run.count("++w.launches;") == 1
    assert "w.launches" not in keys and "rc = run_voxel(h, w, vp, st, false, false);" in keys
    assert "rc = cell_keys_sort(h, vp, 1.0f / cell, st);" in run
    assert "constexpr int ROR_THREADS = 256;" in ror and E.ROR_THREADS == 256
    assert "constexpr unsigned long long LONG_GAP = 2048;" in ror and "to - from >= LONG_GAP" in ror and E.ROR_LONG_GAP == 2048
    assert "constexpr int LIST = 32;" in ror and E.ROR_LIST == 32
    assert "0x28215u" in ror and "0x22161u" in ror and (E.ROR_ROW_DZ, E.ROR_ROW_DY) == (0x28215, 0x22161)
    assert E.ror_rows() == [(0, 0), (0, -1), (0, 1), (-1, 0), (1, 0), (-1, -1), (-1, 1), (1, -1), (1, 1)]
    assert "dv > (1ll << 21)" in vox and "1073741824.f" in vox
    assert "if (g.zero_keys) return;" in ror and "w.plan_error == CM_DEV_E_KEY_RANGE" in keys


def _two_apart(x, pairs, cell):
    c = E.ror_cells(x, cell)
    return (np.abs(c[pairs[:, 0]] - c[pairs[:, 1]]) >= 2).any(axis=1)


@pytest.mark.parametrize("radius", E.ROR_RADII + (E.ROR_RADIUS_TIGHT,))
def test_margin_pairs_stay_one_cell_apart(radius):
    """N-margin: with the shipped margin no neighbour pair is two cells apart on any axis, up to |cell index| 2^14 - 1 on
    both signs, on both sides of the strict rule. Without the margin (cell = radius) the radius 0.45 puts more than 1 % of
    the neighbour pairs two cells apart -- pairs the nine rows would not see. For the other radii the float32 cell is not
    below the radius and the computed planes are never closer than it: there the margin is not what keeps them apart."""
    for sign in (1, -1):
        x = E.margin_cloud(radius, sign)
        pairs = E.ror_pairs(x, radius)
        designed = pairs[(pairs[:, 1] - pairs[:, 0] == 1) & (pairs[:, 0] % 2 == 0)]
        assert 0.4 * len(x) / 2 < len(designed) < len(x) / 2   # some designed pairs fall just outside the radius
        assert not _two_apart(x, pairs, E.ror_cell(radius)).any()
        without = _two_apart(x, pairs, E.ror_cell(radius, margin=False)).mean()
        if radius == E.ROR_RADIUS_TIGHT and sign > 0:
            assert without >= 0.01, without
        elif radius != E.ROR_RADIUS_TIGHT:
            assert without == 0.0
        c = E.ror_cells(x, E.ror_cell(radius))
        assert (c.max() if sign > 0 else -c.min()) == E.ROR_BOUND - 1 and np.abs(c).max() == E.ROR_BOUND - 1
        assert (c == 0).any()
        plan = E.ror_plan([x], radius)
        assert not plan["bound_error"] and not plan["plan_error"]


def _assert_neighbours_searched(clouds, radius):
    plan = E.ror_plan(clouds, radius)
    for c, pt in zip(clouds, plan["points"]):
        pairs = E.ror_pairs(c, radius)
        for a, b in ((0, 1), (1, 0)):
            seg = pt["seg"][pairs[:, a]]
            kb = pt["key"][pairs[:, b]][:, None]
            assert ((seg[:, :, 0] <= kb) & (kb <= seg[:, :, 1])).any(axis=1).all()
    return plan


@pytest.mark.parametrize("name", sorted(E.ror_cases()))
def test_every_counted_neighbour_lies_in_the_searched_rows(name):
    """For every edge cloud the run must succeed: each neighbour the oracle counts has its key in one of the nine row
    segments the point searches, and with the table no read leaves it ([k_lo, k_hi + 1] <= table_keys)."""
    clouds, radius, _ = E.ror_cases()[name]
    plan = _assert_neighbours_searched(clouds, radius)
    assert not plan["plan_error"] and not plan["bound_error"]
    if plan["table"]:
        assert max(int(p["max_read"].max(initial=-1)) for p in plan["points"]) <= plan["table_keys"]


def test_bound_clouds_sit_on_the_bound():
    """N-bound: the largest |cell index| is exactly 2^14 - 1 (accepted) or 2^14 (refused by the count kernel), on each axis
    and sign; the grid itself stays in range."""
    r = float(np.float32(0.15))
    for axis in range(3):
        for sign in (1, -1):
            for idx, refused in ((E.ROR_BOUND - 1, False), (E.ROR_BOUND, True)):
                x = E.bound_cloud(r, axis, sign * idx)
                c = E.ror_cells(x, E.ror_cell(r))
                assert (c[:, axis].max() if sign > 0 else -c[:, axis].min()) == idx
                assert np.abs(np.delete(c, axis, axis=1)).max() < 4
                plan = E.ror_plan([x], r)
                assert plan["worst"] == idx and plan["bound_error"] == refused and not plan["plan_error"]


@pytest.mark.parametrize("name", ["range:wide", "range:far", "range:multi"])
def test_out_of_range_grids_read_past_the_table_unless_refused(name):
    """N-range: the grid of an out-of-range cloud is keyed as one cell but keeps its real div_b. The count as it was
    before the host check (fixed=False) then reads table entries far past table_keys -- the defect. The fixed library
    refuses the call before the table and the count, and would not count such a frame at all."""
    clouds, r = E.ror_refused_cases()[name]
    before = E.ror_plan(clouds, r, fixed=False)
    assert before["plan_error"] and before["table"]
    worst_read = max(int(p["max_read"].max(initial=-1)) for p in before["points"])
    assert worst_read > before["table_keys"], (worst_read, before["table_keys"])
    if name == "range:wide":
        g = before["grids"][0]
        assert g["zero_keys"] and tuple(g["div"]) == (2656291, 2656291, 1) and before["idx_bits"] == 0
        assert before["table_keys"] == 1 and worst_read == 2656293
    after = E.ror_plan(clouds, r)
    assert after["refused"] and all((p["max_read"] < 0).all() for p in after["points"])


def test_gap_layouts_hit_the_table_edges():
    """N-gap: the sorted keys give the gap lengths around LONG_GAP, 31 / 32 / 33 long gaps in one CTA of k_ror_table,
    M % 256 in {0, 1, 255} (thread M fills the top gap, alone in its CTA when M % 256 == 0) and a long empty range above
    the largest key."""
    r = float(np.float32(0.15))
    for kind in E.GAP_KINDS:
        x = E.gap_cloud(r, E.gap_steps(kind))
        plan = E.ror_plan([x], r)
        keys = np.sort(plan["points"][0]["key"])
        assert len(np.unique(keys)) == len(keys) and plan["table"]
        to_minus_from = np.diff(keys) - 1
        long_at = np.nonzero(to_minus_from >= E.ROR_LONG_GAP)[0] + 1        # element that fills it
        if kind == "edge":
            assert {2046, 2047, 2048, 2049} <= set(to_minus_from.tolist())
        if kind.startswith("cta"):
            per_cta = np.bincount(long_at // E.ROR_THREADS)
            assert per_cta[1] == int(kind[3:]) and (np.delete(per_cta, 1) <= E.ROR_LIST).all()
        if kind.startswith("m"):
            assert len(keys) == int(kind[1:]) and len(keys) % 256 in (0, 1, 255)
        assert plan["table_keys"] - keys[-1] >= 1000


def test_width_layouts_hit_every_pass_count_and_the_table_bound():
    """N-width: 1-4 radix passes with 32-bit keys and 5-6 with 64-bit ones (both parities on both widths), and the
    table / binary-search boundary at idx_bits 25 / 26 for one cloud and 24 / 25 for two."""
    cases = E.ror_cases()
    got = {}
    for name in [n for n in cases if n.startswith("width:")]:
        clouds, r, _ = cases[name]
        p = E.ror_plan(clouds, r)
        got[name] = (p["idx_bits"], p["key_bytes"], p["passes"], p["table"])
    assert {(b, p) for (_, b, p, _) in got.values()} >= {(4, 1), (4, 2), (4, 3), (4, 4), (8, 5), (8, 6)}
    assert got["width:25"][::3] == (25, True) and got["width:26"][::3] == (26, False)
    assert got["width:2x24"][::3] == (24, True) and got["width:2x25"][::3] == (25, False)


def test_count_layouts():
    """N-count: a hot cell of 2000+ points with exact duplicates, flat grids (d = 1 on one and two axes), a single-cell
    cloud, non-finite rows, and frames whose last and first key cells are next to each other in key order."""
    r = float(np.float32(0.15))
    cell = E.ror_cell(r)
    hot = E.count_cloud(r, "hot")
    _, counts = np.unique(E.ror_cells(hot, cell), axis=0, return_counts=True)
    assert counts.max() >= 2000 and len(np.unique(hot[:, :3], axis=0)) < len(hot)
    assert (E.ror_grid(E.count_cloud(r, "flat1"), cell)["div"] == 1).sum() == 1
    assert (E.ror_grid(E.count_cloud(r, "flat2"), cell)["div"] == 1).sum() == 2
    assert (E.ror_grid(E.count_cloud(r, "single"), cell)["div"] == 1).all()
    assert (~np.isfinite(E.count_cloud(r, "nonfinite")[:, :3]).all(axis=1)).sum() == 60
    clouds = E.row_end_clouds(r)
    plan = E.ror_plan(clouds, r)
    cells = 8 * 4 * 2
    for f, pt in enumerate(plan["points"]):
        k = pt["key"] - (f << plan["idx_bits"])
        assert k.min() == 0 and k.max() == cells - 1 and E.ror_grid(clouds[f], cell)["div"].tolist() == [8, 4, 2]
        c0 = pt["cells"][:, 0]
        assert (c0 == 0).sum() >= 3 and (c0 == 7).sum() >= 3
    assert plan["idx_bits"] == 6 and cells == 1 << plan["idx_bits"]   # the last cell of frame f is key (f + 1) << 6 minus 1


@pytest.mark.parametrize("name", [n for n in sorted(E.ror_cases()) if not n.startswith("margin:") or n.startswith("margin:0.15f")])
def test_ror_oracle_agrees_with_the_brute_force_count(oracle, name):
    """The C++ oracle (cmo_radius_outlier) against the O(n^2) numpy count on every N cloud small enough."""
    clouds, r, min_pts = E.ror_cases()[name]
    for c in clouds:
        k = E.ror_brute_count(c, r)
        fin = np.isfinite(c[:, :3]).all(axis=1)
        for m in min_pts:
            for neg in (False, True):
                want = np.nonzero(fin & ((k <= m) if neg else (k > m)))[0]
                got = oracle.radius_outlier(c, r, m, neg)
                assert len(got) == len(want) and (got == want).all(), (m, neg)
