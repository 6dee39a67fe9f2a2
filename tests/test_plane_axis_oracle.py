"""CPU tests of the axis-constrained plane models (SACMODEL_PERPENDICULAR_PLANE / SACMODEL_PARALLEL_PLANE):
the C++ statement (tests/plane_axis_oracle.cpp) against the numpy restatement (tests/plane_axis_np.py), the library's float cutoffs (cm_plane_axis_rule)
against PCL's double predicate on windows of floats around every cutoff, and the scene the models exist for."""
import json
import math
import os

import numpy as np
import pytest

import plane_axis as A
from cloud_merger_b200 import CloudMerger, _lib
import plane_axis_np as N
import plane_axis_oracle as PO
from oracle import np_oracle as NP

CASES = A.axis_plane_cases()
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "plane_axis.json")


def _expected_inliers(cloud, w_np, final_coeff, case, order, optimize):
    """What selectWithinDistance keeps at the end: nothing when the final model fails the axis test."""
    if not w_np["found"] or not w_np["best_valid"]:
        return np.zeros(0, np.int64)
    c = final_coeff if optimize else w_np["coeff"]
    if not N.plane_model_valid(c, case["model"], case["axis"], case["eps_angle"], order):
        return np.zeros(0, np.int64)
    return np.flatnonzero(NP.plane_inlier_mask(cloud, c, case["threshold"], order))


@pytest.mark.parametrize("family", ["A-bound", "A-nan", "A-none", "A-refit", "A-free", "A-axis", "A-multi"])
def test_oracle_and_numpy_restatement_agree(family):
    for name, case in sorted(CASES.items()):
        if not name.startswith(family + ":"):
            continue
        for cloud in case["clouds"]:
            for order in case["orders"]:
                w_np = N.plane_ransac(cloud, case["threshold"], case["probability"], case["max_iterations"], case["seed"], order,
                                      case["model"], case["axis"], case["eps_angle"])
                for optimize in case["optimizes"]:
                    what = "%s, order %d, optimize %d" % (name, order, optimize)
                    w = PO.plane_ransac_model(cloud, case["threshold"], case["probability"], case["max_iterations"],
                                                  optimize, case["seed"], order, case["model"], case["axis"], case["eps_angle"])
                    for key in ("found", "iterations", "draws", "best_count", "rejected"):
                        assert w[key] == w_np[key], (what, key, w[key], w_np[key])
                    if w["found"]:
                        assert (w["sample"] == w_np["sample"]).all(), what
                        assert w["coeff_ransac"].tobytes() == w_np["coeff"].tobytes(), what
                    want = _expected_inliers(cloud, w_np, w["coeff"], case, order, optimize)
                    assert (w["inliers"].astype(np.int64) == want).all() and len(w["inliers"]) == len(want), what


def test_cases_reach_their_edges():
    """Each family does what it is there for (so that a library that got it wrong would fail on the GPU)."""
    flips = {}
    for name, c in CASES.items():
        cl = c["clouds"][0]
        args = (c["threshold"], c["probability"], c["max_iterations"], True, c["seed"], c["orders"][0], c["model"], c["axis"])
        w = PO.plane_ransac_model(cl, *args, c["eps_angle"])
        if "draw_valid" in c:   # the boundary draw passes at its own angle and fails one double below
            s = A.P.draw_stream(len(cl), c["seed"], c["draw"] + 1)[c["draw"]]
            good, m = NP.plane_of_sample(cl[s[0]], cl[s[1]], cl[s[2]], c["orders"][0])
            assert good and N.plane_model_valid(m, c["model"], c["axis"], c["eps_angle"], c["orders"][0]) == c["draw_valid"], name
            if c["model"] == A.PERP:   # the second normalize decides, on the side of 0 the case names
                d2 = N.plane_axis_dot(m, A.PERP, c["axis"], c["orders"][0])
                d1 = N.plane_axis_dot(m, A.PAR, c["axis"], c["orders"][0])
                assert d1 != d2 and c["draw_sign"] * float(d2) > 0, name
                one = not N.perpendicular_angle(d1) > c["eps_angle"]
                flips.setdefault(name.rsplit(":", 1)[0], []).append(one != c["draw_valid"])
        if c.get("no_valid"):
            assert w["found"] and w["iterations"] == c["max_iterations"] + 1 == w["rejected"] and len(w["inliers"]) == 0, name
        if c.get("refit_leaves"):
            assert w["found"] and w["best_count"] > 100 and len(w["inliers"]) == 0, name
        if c.get("same_as_plane"):
            p = PO.plane_ransac_model(cl, *args[:-2], 0, A.Z, 0.0)
            assert w["rejected"] == 0 and w["iterations"] == p["iterations"] and (w["inliers"] == p["inliers"]).all(), name
            assert w["coeff"].tobytes() == p["coeff"].tobytes(), name
        if name.startswith("A-nan"):
            r = N.plane_ransac(cl, *args[:3], c["seed"], c["orders"][0], c["model"], c["axis"], c["eps_angle"])
            assert r["rejected"] < r["iterations"], name
    # with one normalize only, the boundary draw would decide the other way at eps "at" or at eps "below"
    assert len(flips) == 6 and all(any(v) for v in flips.values()), flips
    rej = {n: PO.plane_ransac_model(c["clouds"][0], c["threshold"], c["probability"], c["max_iterations"], False, c["seed"],
                                        c["orders"][0], c["model"], c["axis"], c["eps_angle"])["rejected"]
           for n, c in CASES.items() if n.startswith("A-bound")}
    for n in rej:
        if n.endswith(":at"):
            assert rej[n[:-3] + ":below"] == rej[n] + 1, n   # exactly the boundary draw flips


def test_plane_model_is_the_plane_oracle(oracle):
    """With SACMODEL_PLANE the loop of tests/plane_axis_oracle.cpp is oracle/cm_oracle.cpp's cmo_plane_ransac."""
    for name, c in sorted(CASES.items()):
        for cloud in c["clouds"]:
            for optimize in c["optimizes"]:
                args = (c["threshold"], c["probability"], c["max_iterations"], optimize, c["seed"], c["orders"][0])
                a, b = PO.plane_ransac_model(cloud, *args), oracle.plane_ransac(cloud, *args)
                for key in ("found", "iterations", "draws", "best_count"):
                    assert a[key] == b[key], (name, key)
                assert a["rejected"] == 0 and (a["sample"] == b["sample"]).all(), name
                assert a["coeff_ransac"].tobytes() == b["coeff_ransac"].tobytes(), name
                assert a["coeff"].tobytes() == b["coeff"].tobytes() and (a["inliers"] == b["inliers"]).all(), name


def _perp_valid(d, eps):
    rad = float(d)
    rad = -1.0 if rad < -1.0 else 1.0 if rad > 1.0 else rad
    a = abs(math.acos(rad))
    return not min(a, math.pi - a) > eps


def _window(center_bits, half):
    u = np.arange(int(center_bits) - half, int(center_bits) + half + 1, dtype=np.int64)
    return u


def _check_perp_side(rule, eps, cutoff, positive, half=1 << 20):
    """Every float of the window on one side of 0 decides as PCL's double predicate does."""
    mag = int(np.float32(abs(cutoff)).view(np.uint32))
    u = _window(mag, half)
    u = u[(u >= 0) & (u <= 0x3F800000 + 4)]
    d = u.astype(np.uint32).view(np.float32)
    if not positive:
        d = -d
    d64 = np.clip(d.astype(np.float64), -1.0, 1.0)
    with np.errstate(invalid="ignore"):
        a = np.arccos(d64)
    a = np.minimum(a, math.pi - a)
    want = ~(a > eps)
    near = np.abs(a - eps) <= 1e-12 * max(eps, 1e-300) + 1e-300   # decide these with the libm acos, as PCL does
    for i in np.flatnonzero(near):
        want[i] = _perp_valid(d[i], eps)
    if rule["test"] == 0:
        got = np.ones(len(d), bool)
    else:
        got = (d <= rule["c_neg"]) | (d >= rule["c_pos"])
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, (eps, positive, d[bad[:4]])


@pytest.mark.parametrize("eps", [1e-300, 1e-30, 1e-7, math.radians(0.5), math.radians(10.0), 1.0, 1.5, 1.5707963,
                                 A.prev_double(math.pi / 2), math.pi / 2, 2.0])
def test_perpendicular_cutoffs_match_the_double_predicate(eps):
    rule = CloudMerger.plane_axis_rule(A.PERP, A.Z, eps)
    if eps >= math.pi / 2:
        assert rule["test"] == 0
    c_pos = rule["c_pos"] if rule["test"] else np.float32(0)
    c_neg = rule["c_neg"] if rule["test"] else np.float32(-0.0)
    _check_perp_side(rule, eps, c_pos, True)
    _check_perp_side(rule, eps, c_neg, False)


@pytest.mark.parametrize("eps", [1e-300, 1e-30, 1e-7, math.radians(10.0), 1.0, A.prev_double(math.pi / 2), math.pi / 2, 2.0, 4.0])
def test_parallel_cutoff_matches_the_double_predicate(eps):
    rule = CloudMerger.plane_axis_rule(A.PAR, A.Z, eps)
    assert rule["test"] == A.PAR
    s = abs(math.sin(eps))
    u = _window(int(rule["f_plus"].view(np.uint32)), 1 << 20)
    u = u[(u >= 0) & (u < 0x7F800000)]
    d = u.astype(np.uint32).view(np.float32)
    for sign in (1, -1):
        dd = (sign * d).astype(np.float32)
        want = ~(np.abs(dd).astype(np.float64) > s)
        got = ~(np.abs(dd) >= rule["f_plus"])
        assert (got == want).all(), eps


def test_rule_settings_and_axis():
    for eps in (0.0, -1.0, float("nan")):
        for m in (A.PERP, A.PAR):
            assert CloudMerger.plane_axis_rule(m, A.Z, eps)["test"] == 0
    assert CloudMerger.plane_axis_rule(A.PLANE, A.Z, 0.3)["test"] == 0
    r = CloudMerger.plane_axis_rule(A.PERP, (0.0, 0.0, 5.0), 0.3)
    assert r["axis"].tolist() == [0.0, 0.0, 1.0, 0.0]
    r = CloudMerger.plane_axis_rule(A.PERP, (0.0, 0.0, 1e-30), 0.3)   # squared norm underflows: not normalized
    assert r["axis"][2] == np.float32(1e-30)
    for order in (0, 1, 2):
        r = CloudMerger.plane_axis_rule(A.PAR, (0.3, 0.1, 2.0), 0.3, order)
        assert r["axis"].tobytes() == N.normalize4([0.3, 0.1, 2.0, 0.0], order).tobytes()
    with pytest.raises(Exception) as e:
        CloudMerger.plane_axis_rule(3, A.Z, 0.3)
    assert getattr(e.value, "code", None) == _lib.CM_E_INVALID


def test_wall_zone_scene():
    """A zone whose wall holds more points than its ground: PLANE returns the wall, PERPENDICULAR at 10 degrees the
    ground, PARALLEL at 10 degrees a vertical plane."""
    x = A.wall_zone(seed=3)
    plane = PO.plane_ransac_model(x, 0.3, model=A.PLANE)
    perp = PO.plane_ransac_model(x, 0.3, model=A.PERP, eps_angle=A.TEN_DEG)
    par = PO.plane_ransac_model(x, 0.3, model=A.PAR, eps_angle=A.TEN_DEG)
    assert abs(plane["coeff"][0]) > 0.99 and len(plane["inliers"]) > 1000
    assert abs(perp["coeff"][2]) > 0.99 and 500 < len(perp["inliers"]) < 1000
    assert abs(par["coeff"][2]) < 0.2


def test_golden_file():
    """tests/golden/plane_axis.json (tests/golden/make_plane_axis.py): the C++ statement's answers, kept to catch drift."""
    g = json.load(open(GOLDEN))
    for e in g["cases"]:
        x = A.wall_zone(*e["scene"]) if e["scene_kind"] == "wall" else A.walls_only(*e["scene"])
        w = PO.plane_ransac_model(x, e["threshold"], e["probability"], e["max_iterations"], e["optimize"], 12345,
                                      e["sum_order"], e["model"], e["axis"], e["eps_angle"])
        for key in ("found", "iterations", "draws", "best_count", "rejected"):
            assert w[key] == e[key], (e["name"], key)
        assert w["coeff"].view(np.uint32).tolist() == e["coeff_bits"], e["name"]
        assert len(w["inliers"]) == e["n_inliers"], e["name"]
