"""CPU checks of the statistical outlier removal's edge inputs (tests/sor_edges.py, family S): the restated constants
match the sources, the plan restatement puts every case where it was built to be, the search model equals the exact
k nearest neighbours on every case and stops where each bound case was built to stop, the cases discriminate (a search
without eps, a search stopping one step early, a parallel sum where the serial chain is required would all give other
values), the numpy and C++ restatements agree, and the GPU cases stay inside a cost budget. Also pins the cost cliff of
one cell edge for clouds of very different density."""
import math
import os
import re

import numpy as np
import pytest

import sor_edges as S
import sor_np
import sor_oracle
from helpers import host_function

SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "cloud_merger_b200", "csrc")
CASES = S.sor_cases()
F32 = np.float32


def _src(name):
    with open(os.path.join(SRC, name)) as f:
        return f.read()


def _plan(case, table=True):
    return S.sor_plan(case["clouds"], case["mean_k"], case.get("cell"), table)


def _valid(c, mean_k):
    return int(np.isfinite(np.asarray(c, F32)[:, :3]).all(axis=1).sum()) > mean_k


def test_sor_constants_match_the_shared_front_end():
    """The S-family restatement mirrors the kernels' constants; a retune must fail here rather than miss the edges."""
    sor, api, vox = _src("cm_statistical.cu"), _src("cm_api.cu"), _src("cm_voxel.cu")
    body, front, keys, table = (host_function(f) for f in ("statistical_outlier_run", "cell_keys_begin", "cell_keys_sort",
                                                           "enqueue_cell_table"))
    assert "s.mean_k + 1 <= 32 ? 1 : s.mean_k + 1 <= 64 ? 2 : 4" in sor and S.SOR_NS_LIMITS == (32, 64)
    assert re.search(r"constexpr int SOR_WARPS = (\d+);", sor).group(1) == str(S.SOR_WARPS)
    assert re.search(r"constexpr int SUM_THREADS = (\d+);", sor).group(1) == str(S.SUM_THREADS)
    assert re.search(r"constexpr int SERIAL_TILE = (\d+);", sor).group(1) == str(S.SERIAL_TILE)
    assert "r += max(1ll, r >> 1);" in sor and S.growth(30) == [0, 1, 2, 3, 4, 6, 9, 13, 19, 28]
    assert "((double)mb + 1.0) * 0x1p-23 * (1.0 + 0x1p-20) + 0x1p-140" in sor
    assert (S.EPS_REL, S.EPS_MARGIN, S.EPS_ABS) == (2.0 ** -23, 1.0 + 2.0 ** -20, 2.0 ** -140)
    assert "const double bound = a * a * (1.0 - 0x1p-20);" in sor and "bound >= 0x1p-100 && bound >= (double)thr" in sor
    assert (S.BOUND_FACTOR, S.BOUND_FLOOR) == (1.0 - 2.0 ** -20, 2.0 ** -100)
    assert "if (thr <= 0.f) break;" in sor and "const double m = (double)r - eps;" in sor
    assert "mag / 1048576.0, e[a] / 524288.0" in api and (S.FLOOR_MAG, S.FLOOR_EXTENT) == (2.0 ** 20, 2.0 ** 19)
    assert "floor_edge * (1.0 + 1.0 / 1024.0)" in api and S.FLOOR_MARGIN == 1.0 + 1.0 / 1024.0
    assert "std::min(std::max(edge, 1e-30), 1e36)" in api and (S.EDGE_MIN, S.EDGE_MAX) == (1e-30, 1e36)
    assert "const float inv = (float)(1.0 / sor_cell_edge(" in body and "rc = cell_keys_sort(h, vp, inv, st);" in body
    assert ("w.plan_idx_bits <= 25 && ((uint64_t)n_clouds << w.plan_idx_bits) <= (1ull << 25) &&\n      "
            "!getenv(no_table_env)") in table and S.TABLE_LOG2 == 25
    assert 'enqueue_cell_table(h, vp, "CM_SOR_NO_TABLE", rp, st)' in body
    assert "dv > (1ll << 21)" in vox and "1073741824.f" in vox
    # the launches cm_launch_count reports for the call (sor_plan's "launches"): a bounding box per cloud and the table in
    # the shared front end, the search, sums and select in the run
    assert front.count("++w.launches;") == 1 and table.count("++w.launches;") == 1
    assert body.count("++w.launches;") == 0 and body.count("w.launches += 2;") == 2
    assert "w.launches" not in keys and "rc = run_voxel(h, w, vp, st, false, false);" in keys
    assert "zone_run(h, pts, n_points, st, true, n_clouds)" in body


@pytest.mark.parametrize("name", sorted(CASES))
def test_plan_puts_every_case_where_it_was_built(name):
    """Finite input never meets CM_E_KEY_RANGE (DESIGN section 8), and every S-plan case lands on its key width, pass
    count, frame bits, table decision, floor or clamp."""
    case = CASES[name]
    plan = _plan(case)
    assert not plan["key_range"], name
    assert plan["launches"] == sum(1 for c in case["clouds"] if len(c)) + 6 + plan["passes"] + int(plan["table"])
    if "passes" in case:
        assert plan["passes"] == case["passes"] and plan["frame_bits"] == 0
        assert plan["key_bytes"] == (4 if case["passes"] <= 4 else 8)
    if name in ("plan:passes:4", "plan:passes:5"):
        assert plan["total_bits"] == (32 if name.endswith("4") else 33)
    if name.startswith("plan:frames"):
        sentinel = name.endswith("sentinel")
        assert plan["idx_bits"] == 12 and plan["frame_bits"] == (5 if sentinel else 4)
        assert plan["passes"] == (3 if sentinel else 2) and plan["table"]
    if name.startswith("plan:table"):
        n, bits = (int(v) for v in name.split(":")[2].split("x"))
        assert len(case["clouds"]) == n and plan["idx_bits"] == bits
        assert (n << bits) == (1 << 25) * (2 if bits in (22, 26) else 1)
        assert plan["table"] == ((n << plan["idx_bits"]) <= 1 << 25)
        assert not _plan(case, table=False)["table"]
    if "floor" in case:
        assert plan["floor_binds"] and plan["edge"] == plan["floor"] > float(case["cell"])
        mn = np.concatenate(case["clouds"])[:, :3].astype(np.float64)
        ext = (mn.max(axis=0) - mn.min(axis=0)).max() / S.FLOOR_EXTENT
        mag = np.abs(mn).max() / S.FLOOR_MAG
        assert (ext > mag) == (case["floor"] == "extent")
    if "clamp" in case:
        assert plan["clamp"] == case["clamp"]
        assert np.isfinite(plan["inv"]) and plan["inv"] >= np.finfo(F32).tiny
    if name == "plan:passes:8":
        assert plan["total_bits"] == 57 and all(abs(int(d) - 523777) <= 2 for d in plan["grids"][0]["div"])


def test_plan_floor_through_utm_magnitude_sets_a_half_cell_eps():
    """At |x * inv| ~ 2^20 the bound's eps reaches 1/8 cell: the regime the eps term exists for."""
    plan = _plan(CASES["plan:floor:utm"])
    eps = S.search_eps(plan["grids"][0])
    assert 0.12 < eps < 0.13 and max(abs(int(v)) for v in plan["grids"][0]["max_b"]) > 1_040_000


@pytest.mark.parametrize("name", sorted(CASES))
def test_search_model_equals_exact_knn(name):
    """sor_search (k_sor_knn's cubes, bound and stops) keeps exactly the mean_k + 1 smallest float squared distances."""
    case = CASES[name]
    plan = _plan(case)
    for f, c in enumerate(case["clouds"]):
        if not _valid(c, case["mean_k"]):
            continue
        got = S.sor_search(c, plan, case["mean_k"], frame=f)
        assert (got["stop"] >= 0).all()
        fin = np.isfinite(c[:, :3]).all(axis=1)
        want = sor_np.knn_sq(np.ascontiguousarray(c[fin, :3]), case["mean_k"] + 1)
        same = (got["knn"].view(np.uint32) == want.view(np.uint32))
        assert same.all(), "%s cloud %d: %d points differ" % (name, f, int((~same.all(axis=1)).sum()))


def test_search_model_sees_the_eps_term():
    """S-bound (b): without eps the model stops at r_p with the filler instead of the decoy on every far case -- so these
    cases fail a kernel that dropped eps -- and with eps it matches the exact neighbours (previous test)."""
    far = [n for n in CASES if n.startswith("bound:far:")]
    assert len(far) == len(S.BOUND_RS) - 1
    for name in far:
        case = CASES[name]
        plan = _plan(case)
        c = case["clouds"][0]
        want = sor_np.knn_sq(np.ascontiguousarray(c[:, :3]), case["mean_k"] + 1)
        wrong = S.sor_search(c, plan, case["mean_k"], eps_scale=0.0)
        assert wrong["stop"][0] == case["r_p"], name
        assert not (wrong["knn"][0] == want[0]).all(), name
        cell = S.cells_of(c[:, :3], plan["inv"])
        assert cell[0, 0] == 2 ** 19 - 1 and cell[case["decoys"][0][0], 0] == 2 ** 19 + case["r_p"]
        # the decoy's exact offset is below r_p cells: fl(x * inv) rounded it onto the next cell plane
        dx = (float(c[S.BOUND_K, 0]) - float(c[0, 0])) * float(plan["inv"])
        assert dx < case["r_p"], (name, dx)


@pytest.mark.parametrize("name", sorted(n for n in CASES if n.startswith("bound:")))
def test_bound_cases_stop_where_built(name):
    """Every query of an S-bound case stops at the first growth step past r_p whose bound reaches its k-th value; its
    decoy lies r_p + 1 cells away (outside the cube r_p) and is one of its exact neighbours, so a search that stopped at
    r_p -- one step early -- would keep the filler and give another distance."""
    case = CASES[name]
    plan = _plan(case)
    r_p = case["r_p"]
    for f, c in enumerate(case["clouds"]):
        got = S.sor_search(c, plan, case["mean_k"], frame=f)
        cells = S.cells_of(c[:, :3], plan["inv"])
        want = sor_np.knn_sq(np.ascontiguousarray(c[:, :3]), case["mean_k"] + 1)
        for qi, di in zip(case["queries"][f], case["decoys"][f]):
            assert got["stop"][qi] == S.built_stop(case, plan, f, qi) > r_p, (name, f, qi, got["stop"][qi])
            assert np.abs(cells[di] - cells[qi]).max() == r_p + 1, (name, f, qi)
            d = sor_np._sq_dist(c[qi:qi + 1, :3], c[None, di:di + 1, :3])[0, 0]
            assert d <= want[qi, -1], (name, f, qi)   # the decoy is one of q's mean_k + 1 nearest
            filler = sor_np._sq_dist(c[qi:qi + 1, :3], c[None, di + 1:di + 2, :3])[0, 0]
            assert filler > want[qi, -1] and np.abs(cells[di + 1] - cells[qi]).max() <= r_p, (name, f, qi)


def test_bound_cases_cover_every_direction_and_clipped_cubes():
    plan = _plan(CASES["bound:near:4"])
    g = plan["grids"][0]
    assert len(S.directions()) == 26 and all(int(d) < 2 * 4 + 5 for d in g["div"][1:])   # y, z: clipped cubes
    for f in range(6):
        pc = _plan(CASES["bound:corner:4"])
        cq = S.cells_of(CASES["bound:corner:4"]["clouds"][f][:1, :3], pc["inv"])[0] - pc["grids"][f]["min_b"]
        assert (cq == 0).all()   # the query sits in its grid's corner cell


def test_slot_cases_cover_every_slot_layout():
    ks = {CASES[n]["mean_k"] for n in CASES if n.startswith("slots:")}
    assert {S.ns_of(k) for k in ks} == {1, 2, 4}
    assert {31, 32, 63, 64}.issubset(ks)
    for n in CASES:
        if n.startswith("slots:exact:"):
            c = CASES[n]["clouds"][0]
            assert int(np.isfinite(c[:, :3]).all(axis=1).sum()) == CASES[n]["mean_k"] + 1
    for n in ("slots:cells:40", "slots:cells:62", "slots:cells:126"):
        case = CASES[n]
        assert S.fill_crossings(case["clouds"][0], _plan(case), case["mean_k"]) > 0, n


def test_lattice_slot_cases_have_ties_at_the_kth_value():
    for k in (30, 32, 62, 64, 126):
        c = CASES["slots:lattice:%d" % k]["clouds"][0]
        nn = sor_np.knn_sq(np.ascontiguousarray(c[:, :3]), k + 1)
        nxt = sor_np.knn_sq(np.ascontiguousarray(c[:, :3]), k + 2)[:, -1]
        assert (nxt == nn[:, -1]).any(), k


@pytest.mark.parametrize("name", sorted(n for n in CASES if n.startswith(("sums:", "select:"))))
def test_sum_paths_and_discrimination(name):
    """Every S-sums case takes the path it was built for (k_sor_sums' condition restated); where a sum goes serial, the
    serial chain in index order differs from the exact sum, so a kernel that summed in parallel there would fail."""
    case = CASES[name]
    for c in case["clouds"]:
        w = sor_np.sor_cloud(c, case["mean_k"], 1.0)
        p = S.sum_path(w["distances"])
        if "path" in case and len(case["clouds"]) == 1:
            assert p == case["path"], (name, p)
        v = w["distances"].astype(np.float64)
        with np.errstate(over="ignore"):
            v2 = (w["distances"] * w["distances"]).astype(F32).astype(np.float64)
        if not np.isfinite(v2).all():
            assert p == 3
            continue
        if "tight" in case:   # the sum the case puts just over its boundary, small values last
            bit = case["tight"]
            vals, got = (v, w["sum"]) if bit == 1 else (v2, w["sq_sum"])
            assert p & bit and got == sor_np.serial_sum(vals) != math.fsum(vals.tolist()), (name, bit)
        if p == 0 and len(v):   # exact in any order: the parallel result is PCL's
            assert w["sum"] == math.fsum(v.tolist()) and w["sq_sum"] == math.fsum(v2.tolist())


def test_sum_cases_hit_the_exactness_boundary():
    """The just-over and just-under pairs straddle 2^(53 + e_min) of the sum they test, and the pairs' distances are their
    separations exactly (m * 2^e, m < 2^12, or P1_M whose square rounds to 3 * 2^46)."""
    def units(name, sq):
        d = sor_np.sor_cloud(CASES[name]["clouds"][0], 1, 1.0)["distances"]
        w = (d * d).astype(F32) if sq else d
        e = int(S.lsb_exp(w).min())
        return math.fsum(w.astype(np.float64).tolist()) / math.ldexp(1.0, 53 + e)
    assert units("sums:2p40:4095", False) < 1.0 <= units("sums:2p40:4096", False)
    assert units("sums:sq:under", True) < 1.0 <= units("sums:sq:over", True)
    assert units("sums:both:under", False) < 1.0 <= units("sums:both:over", False)
    assert units("sums:sum:under", False) < 1.0 <= units("sums:sum:over", False) and units("sums:sum:over", True) < 1.0
    m = F32(S.P1_M)
    assert int(S.lsb_exp(F32(m * m))) == 46 and np.sqrt(F32(m * m)) == m
    d = sor_np.sor_cloud(CASES["sums:sum:over"]["clouds"][0], 1, 1.0)["distances"]
    assert d[-1] == F32(S.P1_M * 2.0 ** -23) and d[0] == F32(2.0 ** 22)
    d = sor_np.sor_cloud(CASES["sums:overflow"]["clouds"][0], 1, 1.0)["distances"]
    assert np.isinf(d).sum() == 2 and np.isfinite(d).sum() == 4
    d = sor_np.sor_cloud(CASES["sums:subnormal"]["clouds"][0], 1, 1.0)["distances"]
    assert (F32(d * d) < np.finfo(F32).tiny).all() and (F32(d * d) > 0).all()
    paths = [S.sum_path(sor_np.sor_cloud(c, 1, 1.0)["distances"]) for c in CASES["sums:16-clouds"]["clouds"]]
    assert len(paths) == 16 and set(paths) == {0, 1, 2, 3}


def test_a_finite_distance_has_a_finite_float_square():
    """k_sor_sums flags a finite value with an infinite float square (bad & 2), but no distance is one: the largest finite
    squared distance is FLT_MAX, its root sqrtf(FLT_MAX) = 1.8446743e19 squares to a finite float, and a mean of roots is
    at most their largest -- in float and in double sqrt mode, for every mean_k."""
    fmax = np.finfo(F32).max
    r = np.sqrt(fmax)
    assert r == F32(1.8446743e19) and np.isfinite(F32(r * r))
    for k in range(1, 128):
        for root in (float(r), math.sqrt(float(fmax))):
            s = 0.0
            for _ in range(k):
                s += root
            v = F32(s / k)
            assert v <= r and np.isfinite(F32(v * v)), k


def test_select_cases_put_distances_on_the_threshold():
    w = sor_np.sor_cloud(CASES["select:on-threshold"]["clouds"][0], 1, 0.0)
    assert w["mean"] == 2.0 == w["threshold"] and sorted(w["distances"].tolist()) == [1, 1, 2, 2, 3, 3]
    assert w["keep"].sum() == 4
    neg = sor_np.sor_cloud(CASES["select:on-threshold"]["clouds"][0], 1, 0.0, negative=True)
    assert neg["keep"].sum() == 2
    e = CASES["select:empties"]["clouds"]
    assert [len(c) for c in e][0] == 0 and len(e[2]) == 0 and len(e[-1]) == 0


@pytest.mark.parametrize("name", sorted(CASES))
def test_numpy_and_cpp_restatements_agree(name):
    case = CASES[name]
    for c in case["clouds"]:
        for sm in (0, 1):
            a = sor_np.sor_cloud(c, case["mean_k"], case.get("std_mul", 1.0), sqrt_mode=sm)
            b = sor_oracle.statistical_outlier(c, case["mean_k"], case.get("std_mul", 1.0), sqrt_mode=sm)
            assert (a["distances"].view(np.uint32) == b["distances"].view(np.uint32)).all(), (name, sm)
            assert (a["keep"] == b["keep"]).all() and a["n_valid"] == b["n_valid"] and a["too_few"] == b["too_few"]
            for k in ("mean", "stddev", "threshold", "sum", "sq_sum"):
                assert (np.isnan(a[k]) and np.isnan(b[k])) or a[k] == b[k], (name, k, a[k], b[k])


@pytest.mark.parametrize("name", ["plan:clamp:max", "plan:clamp:min", "sums:overflow", "sums:subnormal",
                                  "sums:subnormal+1", "slots:lattice:64", "bound:far:4", "sums:16-clouds"])
def test_knn_sq_against_brute_force(name):
    """sor_np.knn_sq's cKDTree slack loop against an O(n^2) sort, where infinities, subnormal squares, ties and rounding
    across cell planes are involved."""
    case = CASES[name]
    for c in case["clouds"]:
        fin = np.isfinite(c[:, :3]).all(axis=1)
        p = np.ascontiguousarray(c[fin, :3])
        if len(p) <= case["mean_k"]:
            continue
        with np.errstate(over="ignore", invalid="ignore"):
            brute = np.sort(sor_np._sq_dist(p, np.broadcast_to(p[None], (len(p),) + p.shape)), axis=1)
        want = brute[:, :case["mean_k"] + 1]
        assert (sor_np.knn_sq(p, case["mean_k"] + 1).view(np.uint32) == want.view(np.uint32)).all(), name


@pytest.mark.parametrize("name", sorted(CASES))
def test_cost_guard(name):
    """Every GPU case's search stays inside the budget (row pieces of the worst point and of the whole call)."""
    case = CASES[name]
    worst, total = S.search_cost(case["clouds"], _plan(case), case["mean_k"])
    assert worst <= S.COST_WORST and total <= S.COST_TOTAL, (name, worst, total)


def test_one_cell_edge_for_clouds_of_very_different_density_is_a_cost_cliff():
    """Documented limitation (DESIGN section 8, open): the edge comes from the largest cloud and serves every cloud of the
    call. A 1 M-point 2 m x 2 m patch next to 200 points in a 1 km cube gets a 3.7 mm edge; the sparse cloud then spans
    ~2.7e5 cells per axis, its 10th neighbours lie ~6.5e4 cells out, its searches end at half-width 92170 and its
    median point visits ~6e10 row pieces -- far beyond
    what may run on a GPU. On its own it would get a 132 m edge and a few dozen pieces per point."""
    dense, sparse = S.cliff_clouds()
    plan = S.sor_plan([dense, sparse], 10)
    assert 3.6e-3 < plan["edge"] < 3.8e-3 and not plan["key_range"]
    assert 2.6e5 < int(plan["grids"][1]["div"].max()) < 2.8e5
    kth = np.sqrt(sor_np.knn_sq(np.ascontiguousarray(sparse[:, :3]), 11)[:, -1].astype(np.float64)) / plan["cell"]
    assert 6e4 < np.median(kth) < 7e4                     # cells to the 10th neighbour
    got = S.sor_search(sparse, plan, 10, frame=1)
    assert np.median(got["stop"]) == 92170                # the growth step past it (... 61447, 92170)
    assert 3e10 < np.median(got["pieces"]) < 1e11         # 6.2e10 row pieces for the median point
    assert got["pieces"].sum() > 1e13
    assert np.median(got["pieces"]) > 1000 * S.COST_WORST
    alone = S.sor_plan([sparse], 10)
    assert 120 < alone["edge"] < 140
    assert S.sor_search(sparse, alone, 10)["pieces"].max() < 200
