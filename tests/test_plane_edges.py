"""CPU checks of the RANSAC ground plane's edge inputs (tests/plane_edges.py, family P): the restated constants and the
launch bookkeeping match the sources, every case lands where it was built (draws and iterations on the intended side of
each round edge, per-tile inlier counts, threshold points on the intended side in all three sum orders, d == +-0), the
cases discriminate (zero padding, a rejection limit of 999 or 1001, a pairwise refit sum, `<=`, a threshold without
the nextafter rounding would each change an output), and the C++ and numpy restatements agree where numpy is fast."""
import os
import re
import time

import numpy as np
import pytest

import plane_edges as P
from helpers import host_function
from oracle import np_oracle as npo

SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "cloud_merger_b200", "csrc")
INC = os.path.join(os.path.dirname(SRC), "..", "include", "cloud_merger_gpu.h")
CASES = P.plane_cases()
F32 = np.float32


def _src(name):
    with open(os.path.join(SRC, name)) as f:
        return f.read()


def _run(oracle, case, cloud, optimize=False, order=0):
    return oracle.plane_ransac(cloud, case["threshold"], case["probability"], case["max_iterations"], optimize,
                               case["seed"], order)


def test_plane_constants_match_the_source():
    """The P-family mirrors the kernels' and the host loop's constants; a retune must fail here rather than miss the
    edges."""
    pl, api, kh = _src("cm_plane.cu"), _src("cm_api.cu"), _src("cm_kernels.h")
    run = host_function("plane_ransac_run")
    assert re.search(r"constexpr int PL_THREADS = (\d+);", pl).group(1) == str(P.PL_THREADS)
    assert re.search(r"constexpr int PL_CHUNK = (\d+);", pl).group(1) == str(P.PL_CHUNK)
    assert re.search(r"constexpr int PM_TILE = (\d+);", pl).group(1) == str(P.PM_TILE)
    assert "constexpr int PM_STRIDE = PM_TILE + 20;" in pl and P.PM_STRIDE == P.PM_TILE + 20
    assert "const uint32_t i = blockIdx.x * 256u + threadIdx.x;" in pl and P.SELECT_BLOCK == 256
    assert "const int pairs = (cnt + 31) >> 5;" in pl
    assert pl.count("make_float4(qnan, qnan, qnan, qnan)") == 3   # the score chunk pad and both moments pads
    assert re.search(r"constexpr size_t PLANE_FIRST_BATCH = (\d+);", api).group(1) == str(P.FIRST_BATCH)
    assert re.search(r"constexpr size_t PLANE_SECOND_BATCH = (\d+);", api).group(1) == str(P.SECOND_BATCH)
    assert re.search(r"constexpr size_t PLANE_BATCH = (\d+);", api).group(1) == str(P.BATCH)
    assert "batch = batch == PLANE_FIRST_BATCH ? PLANE_SECOND_BATCH : PLANE_BATCH;" in run
    assert "if (++s.bad_run == %d) s.stop = true;" % P.REJECT_LIMIT in run
    assert "n_in < %d) continue;" % P.REFIT_FLOOR in run
    assert "thr = std::nextafter(thr, std::numeric_limits<float>::infinity());" in run
    assert "< p.threshold" in pl and "< q.threshold" in pl and pl.count("<= q.threshold") + pl.count("<= p.threshold") == 0
    assert "#define CM_MAX_PLANE_CLOUDS (CM_MAX_ZONES / 2)" in kh
    assert int(re.search(r"#define CM_MAX_ZONES (\d+)", open(INC).read()).group(1)) // 2 == P.MAX_CLOUDS
    assert re.search(r"#define CM_ZONE_LAUNCHES (\d+)", kh).group(1) == str(P.ZONE_LAUNCHES)
    # the launches cm_launch_count reports (plane_launches): one score per round, the moments when refitting, the select
    # when there are points, and the compaction's own count
    assert run.count("++launches;") == 3 and "if (n_points) ++launches;" in run
    assert "CM_CUDA(h, launch_plane_score(pp, st));\n    ++launches;" in run
    assert "CM_CUDA(h, launch_plane_moments(ps, (uint32_t)cfg.sum_order, q.acc_dev.get(), st));\n    ++launches;" in run
    assert "if (any_found && cfg.optimize) {" in run
    assert "h->zw.launches += launches;" in run and "h->zone_launches = true;" in run
    assert "z.launches = zp.n_tiles ? CM_ZONE_LAUNCHES : 1;" in host_function("zone_run")
    assert "if (h->zone_launches) return h->zw.launches;" in api


def test_round_bookkeeping():
    assert [P.round_of_draw(d) for d in (0, 1, 32, 33, 288, 289, 1312, 1313, 2336, 2337)] == [0, 1, 1, 2, 2, 3, 3, 4, 4, 5]
    assert P.plane_rounds([0, 33, 1313, 5]) == 4
    assert P.plane_launches([5], True, True, 10) == 1 + 1 + 1 + 3
    assert P.plane_launches([0], True, False, 0) == 0 + 0 + 0 + 1


def test_draw_stream_is_the_oracles_sampler(oracle):
    """draw_stream reproduces the C++ oracle's sample of the best model (the stream does not depend on the data)."""
    x = P._generic(200, 1)
    for m in (0, 5, 40):
        r = oracle.plane_ransac(x, 1e30, 1.0, m, False, 12345, 0)   # every point inside: the first draw stays the best
        assert r["draws"] == m + 1
        assert r["sample"].tolist() == P.draw_stream(200, 12345, 1)[0].tolist()
    # a tiny threshold: the best is the draw with the most points inside; its sample must be one of the stream's draws
    r = oracle.plane_ransac(x, 1e-3, 1.0, 100, False, 7, 0)
    s = P.draw_stream(200, 7, r["draws"])
    assert any((row == r["sample"]).all() for row in s)


@pytest.mark.parametrize("name", sorted(n for n in CASES if n.startswith("P-batch")))
def test_batch_cases_land_on_the_round_edges(oracle, name):
    case = CASES[name]
    r = _run(oracle, case, case["clouds"][0])
    if "draws" in case:   # the cap decides: one before, on and one after each round edge
        assert r["found"] and r["draws"] == r["iterations"] == case["draws"], (name, r["draws"])
        m = case["max_iterations"]
        assert any(m + 1 - e in (-1, 0, 1) for e in P.EDGES)
    else:                 # the stopping rule decides
        assert r["iterations"] == case["iterations"] == r["draws"], (name, r["iterations"])


@pytest.mark.parametrize("d", [33, 289, 1000, 1001])
def test_bad_cases_reject_exactly_until_the_intended_draw(oracle, d):
    case = CASES["P-bad:%d" % d]
    x, off = case["clouds"][0], set(case["off"].tolist())
    s = P.draw_stream(len(x), case["seed"], d)
    assert not any(set(row.tolist()) & off for row in s[:-1]) and set(s[-1].tolist()) & off
    r = _run(oracle, case, x)
    if d <= P.REJECT_LIMIT:
        assert r["found"] and r["draws"] >= d
        # the first good draw is draw d; PCL's loop has scored it, so iteration 1 is over by then
        assert set(r["sample"].tolist()) & off
    else:
        assert not r["found"] and r["draws"] == P.REJECT_LIMIT and r["iterations"] == 0


def test_rejection_limit_discriminates():
    """getSamples gives up after REJECT_LIMIT rejected draws in a row. P-bad:1000's first good draw follows 999
    rejections (a limit of 999 would give up before it) and P-bad:1001's follows 1000 (a limit of 1001 would reach it)."""
    for d in (1000, 1001):
        case = CASES["P-bad:%d" % d]
        off = set(case["off"].tolist())
        s = P.draw_stream(len(case["clouds"][0]), case["seed"], d)
        first = next(i + 1 for i, row in enumerate(s) if set(row.tolist()) & off)
        assert first == d
        found = {lim: first - 1 < lim for lim in (999, 1000, 1001)}
        assert found[999] != found[1000] if d == 1000 else found[1001] != found[1000]


@pytest.mark.parametrize("name", sorted(n for n in CASES if n.startswith("P-chunk")))
def test_chunk_cases(oracle, name):
    """d == +-0 for ground on z = 0, and a zero-filled chunk pad (the kernel scores whole 512-point chunks) would add
    inside points on some case."""
    case = CASES[name]
    x = case["clouds"][0]
    for order in case["orders"]:
        r = _run(oracle, case, x, False, order)
        assert r["found"]
        if case.get("zero_d"):
            assert r["coeff_ransac"][3:].view(np.uint32)[0] in (0, 0x80000000), (name, r["coeff_ransac"])
        pad = (-len(x)) % P.PL_CHUNK
        zero_in = npo.plane_inlier_mask(np.zeros((1, 4), F32), r["coeff_ransac"], case["threshold"], order)[0]
        if case.get("zero_d") and pad:
            assert zero_in   # the padded best count would be best_count + pad: the search changes


def test_zero_padding_discriminates(oracle):
    """A zero-filled chunk pad in k_plane_score would raise the best draw's count by the pad on every P-chunk cloud on
    z = 0 whose size is not a multiple of PL_CHUNK, in every sum order."""
    hit = 0
    for name, case in CASES.items():
        x = case["clouds"][0]
        pad = (-len(x)) % P.PL_CHUNK
        if not case.get("zero_d") or not pad:
            continue
        for order in case["orders"]:
            r = _run(oracle, case, x, False, order)
            c = r["coeff_ransac"]
            assert int(npo.plane_inlier_mask(x, c, case["threshold"], order).sum()) == r["best_count"], name
            padded = np.concatenate([x, np.zeros((pad, 4), F32)])
            assert int(npo.plane_inlier_mask(padded, c, case["threshold"], order).sum()) == r["best_count"] + pad, name
        hit += 1
    assert hit >= 8
    # k_plane_moments: on the noisy origin plane a zero point is inside the RANSAC model; a zero pad would raise n_in
    for n in (200, 300, 1000):
        case = CASES["P-chunk:origin:%d" % n]
        r = _run(oracle, case, case["clouds"][0], False, 0)
        assert npo.plane_inlier_mask(np.zeros((1, 4), F32), r["coeff_ransac"], case["threshold"], 0)[0]
        assert len(case["clouds"][0]) % P.PM_TILE != 0


def _serial(v):
    acc = F32(0)
    for t in v.astype(F32):
        acc = F32(acc + t)
    return acc


def _pairwise(v):
    v = v.astype(F32)
    while len(v) > 1:
        if len(v) % 2:
            v = np.concatenate([v, np.zeros(1, F32)])
        v = (v[0::2] + v[1::2]).astype(F32)
    return v[0] if len(v) else F32(0)


@pytest.mark.parametrize("name", sorted(n for n in CASES if n.startswith("P-tile")))
def test_tile_cases(oracle, name):
    """Per-tile inlier counts as labelled (the RANSAC model's inliers are the ground built into the cloud), and the
    refit floor cases have exactly 3, 4 and 5 inliers."""
    case = CASES[name]
    x = case["clouds"][0]
    r = _run(oracle, case, x, False, 0)
    inl = npo.plane_inlier_mask(x, r["coeff_ransac"], case["threshold"], 0)
    if "floor" in case:
        assert r["best_count"] == case["floor"] == int(case["inliers"].sum())
    else:
        assert (inl == case["inliers"]).all(), name
    if "tile_counts" in case:
        per = [int(inl[t * P.PM_TILE:(t + 1) * P.PM_TILE].sum()) for t in range(len(case["tile_counts"]))]
        assert per == list(case["tile_counts"])
        assert set(P.TILE_COUNTS) <= set(per)
        assert any(per[t] == 0 and per[t - 1] and per[t + 1] for t in range(1, len(per) - 1))


def test_pairwise_refit_sum_discriminates(oracle):
    """The nine refit sums of some P-tile case differ between the serial chain and a pairwise sum (near 1000 m)."""
    differ = 0
    for name, case in CASES.items():
        if not name.startswith("P-tile") or "floor" in case:
            continue
        x = case["clouds"][0]
        r = _run(oracle, case, x, False, 0)
        p = x[npo.plane_inlier_mask(x, r["coeff_ransac"], case["threshold"], 0)]
        terms = [p[:, 0] * p[:, 0], p[:, 0] * p[:, 1], p[:, 0] * p[:, 2], p[:, 1] * p[:, 1], p[:, 1] * p[:, 2],
                 p[:, 2] * p[:, 2], p[:, 0], p[:, 1], p[:, 2]]
        differ += sum(_serial(t) != _pairwise(t) for t in terms)
    assert differ >= 9


@pytest.mark.parametrize("key", sorted(P.THRESHOLDS))
def test_threshold_points_fall_on_the_intended_side(key):
    """With the z = 0 model the distance is exactly |z|: the points at +-t are outside for every float threshold t,
    those at +-nextbelow(t) inside, and the three sum orders agree."""
    thr = P.THRESHOLDS[key]
    x, g = P.thr_cloud(thr)
    z = x[g:, 2]
    c = np.array([0, 0, 1, 0], F32)
    eff = P.effective_threshold(thr)
    want = np.abs(z.astype(np.float64)) < thr   # the double comparison of PCL
    for order in (0, 1, 2):
        m = npo.plane_inlier_mask(x[g:], c, thr, order)
        assert (m == want).all(), (key, order)
        with np.errstate(invalid="ignore"):
            assert (m == (np.abs(z) < eff)).all(), (key, order)   # the kernels' float comparison


def test_threshold_cases_discriminate():
    """`<=` would take the points at t for a float threshold; dropping the nextafter would lose the point at 0.3f."""
    x, g = P.thr_cloud(0.25)
    z = np.abs(x[g:, 2])
    assert ((z <= F32(0.25)) != (z < F32(0.25))).any()
    thr = P.THRESHOLDS["0.3f+ulp"]
    x, g = P.thr_cloud(thr)
    z = np.abs(x[g:, 2])
    assert ((z < P.effective_threshold(thr)) != (z < F32(thr))).any()
    assert (F32(0.3) < P.effective_threshold(thr)) and np.float64(F32(0.3)) < thr


@pytest.mark.parametrize("key", sorted(P.THRESHOLDS))
def test_threshold_case_model_is_the_ground(oracle, key):
    """The search of every P-thr case ends on the z = 0 plane where the threshold lets the ground decide."""
    case = CASES["P-thr:" + key]
    r = _run(oracle, case, case["clouds"][0])
    thr = case["threshold"]
    if np.isfinite(thr) and 0 < thr < 1:
        assert np.abs(r["coeff_ransac"][:2]).max() == 0 and abs(r["coeff_ransac"][2]) == 1, (key, r["coeff_ransac"])
    if thr == thr and thr <= 0 or thr != thr:
        assert r["found"] and r["best_count"] == 0


def test_multi_rounds_case_stops_in_every_round(oracle):
    case = CASES["P-multi:rounds"]
    rounds = sorted({P.round_of_draw(_run(oracle, case, x)["draws"]) for x in case["clouds"]})
    assert rounds == [1, 2, 3, 4]


def test_multi_layouts():
    tiles = P.SELECT_BLOCK, 1024
    for name in ("P-multi:offgrid", "P-multi:empties", "P-multi:tiny", "P-multi:rounds"):
        clouds = CASES[name]["clouds"]
        assert len(clouds) == P.MAX_CLOUDS and (len(clouds[7]) > 0) == (name != "P-multi:empties")
        begin = np.cumsum([len(c) for c in clouds])[:-1]
        if name == "P-multi:offgrid":
            assert all(b % t for b in begin for t in tiles)
    sizes = [len(c) for c in CASES["P-multi:empties"]["clouds"]]
    assert sizes[0] == 0 and sizes[-1] == 0 and 0 in sizes[1:-1]
    assert {1, 2, 3} <= {len(c) for c in CASES["P-multi:tiny"]["clouds"]}


def test_size_cases_cross_the_scan_rounds():
    one, eight = (sum(len(c) for c in case["clouds"]) for case in P.size_cases())
    assert one == P.SCAN_ROUND + 1 and eight == 2 * P.SCAN_ROUND + 777
    assert len(P.size_cases()[1]["clouds"]) == P.MAX_CLOUDS


def test_cpp_and_numpy_restatements_agree_within_budget(oracle):
    """cmo_plane_ransac and np_oracle.plane_ransac (no refit) agree on every case small enough for numpy; the whole
    comparison stays within 60 s of CPU time."""
    t0 = time.process_time()
    done = 0
    for name, case in sorted(CASES.items()):
        for x in case["clouds"]:
            r = _run(oracle, case, x)
            if len(x) * max(r["draws"], 1) > 3e6:
                continue
            w = npo.plane_ransac(x, case["threshold"], case["probability"], case["max_iterations"], case["seed"], 0)
            for k in ("found", "iterations", "draws", "best_count"):
                assert r[k] == w[k], (name, k, r[k], w[k])
            assert (r["sample"] == w["sample"]).all(), name
            if r["found"]:
                assert r["coeff_ransac"].view(np.uint32).tolist() == w["coeff"].view(np.uint32).tolist(), name
            done += 1
    assert done >= 60
    assert time.process_time() - t0 < 60
