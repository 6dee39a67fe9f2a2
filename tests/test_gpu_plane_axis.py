"""GPU parity (-m gpu) of the axis-constrained plane models (tests/plane_axis.py): decisions on the cutoff, NaN models,
searches without a valid model up to the iteration cap, refits that leave the cone, settings that constrain nothing,
degenerate axes, eight-cloud mixes and the reference's four zone tables. Every case runs through plane_ransac,
plane_ransac_multi, dev_plane_ransac and dev_plane_ransac_multi and must be bit-exact against the C++ statement (tests/plane_axis_oracle.cpp);
cm_launch_count must equal the CPU plan (tests/plane_edges.py)."""
import math

import numpy as np
import pytest

import plane_axis as A
import plane_axis_oracle as PO
import plane_edges as P
from cloud_merger_b200 import CloudMerger, synth
from cloud_merger_b200.node import FRONT_PARTS, NodeParams
from helpers import assert_bit_equal, same_floats

pytestmark = pytest.mark.gpu

CASES = A.axis_plane_cases()
CAP = 1 << 16


@pytest.fixture(scope="module")
def cm(gpu_ok):
    with CloudMerger(max_sensors=1, max_points_per_sensor=CAP, max_batch_points=CAP, max_batch_frames=8) as m:
        yield m


def _check(got, ground, rest, cloud, want, what):
    for key in ("found", "iterations", "draws", "best_count", "rejected"):
        assert got[key] == want[key], (what, key, got[key], want[key])
    assert (got["sample"] == want["sample"]).all(), what
    assert same_floats(got["coeff_ransac"], want["coeff_ransac"]), (what, got["coeff_ransac"], want["coeff_ransac"])
    assert same_floats(got["coeff"], want["coeff"]), (what, got["coeff"], want["coeff"])
    gx, gi = ground
    rx, ri = rest
    assert got["n_inliers"] == len(want["inliers"]) == len(gi), what
    assert (np.asarray(gi, np.int64) == want["inliers"]).all(), "inlier set / order of " + what
    others = np.setdiff1d(np.arange(len(cloud)), want["inliers"])
    assert len(ri) == len(others) and (np.asarray(ri, np.int64) == others).all(), "rest set / order of " + what
    assert_bit_equal(gx, cloud[want["inliers"]], "ground coordinates of " + what)
    assert_bit_equal(rx, cloud[others], "rest coordinates of " + what)


def run_four(cm, oracle, case, optimize, order):
    clouds = case["clouds"]
    args = (case["threshold"], case["probability"], case["max_iterations"], optimize, case["seed"], order)
    kw = dict(model=case["model"], axis=case["axis"], eps_angle=case["eps_angle"])
    want = [PO.plane_ransac_model(c, *args, **kw) for c in clouds]
    if case.get("same_as_plane"):   # no constraint: what SACMODEL_PLANE returns, bit for bit
        plain = [PO.plane_ransac_model(c, *args) for c in clouds]
        for w, p in zip(want, plain):
            assert w["rejected"] == 0 and w["iterations"] == p["iterations"] and same_floats(w["coeff"], p["coeff"])
            assert (w["inliers"] == p["inliers"]).all()
    begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    n = int(begin[-1])
    launches = P.plane_launches([w["draws"] for w in want], optimize, any(w["found"] for w in want), n)
    what = "%s, optimize %d, order %d" % (case["name"], optimize, order)
    got = cm.plane_ransac_multi(clouds, *args, **kw)
    assert cm.launch_count() == launches, what + " (multi)"
    for k, (c, g, w) in enumerate(zip(clouds, got, want)):
        _check(g, g["ground"], g["rest"], c, w, "%s, cloud %d (multi)" % (what, k))
    buf = cm.upload(np.ascontiguousarray(np.concatenate(clouds))) if n else None
    got = cm.dev_plane_ransac_multi(buf.ptr if buf else 0, begin, *args, **kw)
    assert cm.launch_count() == launches, what + " (device multi)"
    zones = cm.zone_out()
    for k, (c, g, w) in enumerate(zip(clouds, got, want)):
        gx, gi = zones[2 * k]
        rx, ri = zones[2 * k + 1]
        _check(g, (gx, gi.astype(np.int64) - begin[k]), (rx, ri.astype(np.int64) - begin[k]), c, w,
               "%s, cloud %d (device multi)" % (what, k))
    if buf:
        buf.free()
    for k, (c, w) in enumerate(zip(clouds, want)):
        one = P.plane_launches([w["draws"]], optimize, w["found"], len(c))
        g = cm.plane_ransac(c, *args, **kw)
        assert cm.launch_count() == one, what + " (single)"
        _check(g, g["ground"], g["rest"], c, w, "%s, cloud %d (single)" % (what, k))
        if not len(c):
            continue
        b = cm.upload(c)
        g = cm.dev_plane_ransac(b.ptr, len(c), *args, **kw)
        assert cm.launch_count() == one, what + " (device single)"
        z = cm.zone_out()
        _check(g, z[0], z[1], c, w, "%s, cloud %d (device single)" % (what, k))
        b.free()


@pytest.mark.parametrize("family", ["A-bound", "A-nan", "A-none", "A-refit", "A-free", "A-axis", "A-multi"])
def test_axis_models_match_the_oracle(cm, oracle, family):
    ran = 0
    for name, case in sorted(CASES.items()):
        if not name.startswith(family + ":"):
            continue
        for optimize in case["optimizes"]:
            for order in case["orders"]:
                run_four(cm, oracle, case, optimize, order)
                ran += 1
    assert ran


def test_plane_model_ignores_axis_and_eps(cm, oracle):
    """model = CM_SAC_PLANE: whatever axis and eps_angle hold, the result is the one without them."""
    x = A.wall_zone(seed=61)
    base = cm.plane_ransac(x, 0.3)
    for axis, eps in (((0.0, 0.0, 1.0), A.TEN_DEG), ((0.0, 0.0, 0.0), 0.01), ((1.0, 2.0, 3.0), float("nan")), ((0.0, 0.0, 1.0), -1.0)):
        g = cm.plane_ransac(x, 0.3, model=A.PLANE, axis=axis, eps_angle=eps)
        for key in ("found", "iterations", "draws", "best_count", "rejected", "n_inliers"):
            assert g[key] == base[key], key
        assert same_floats(g["coeff"], base["coeff"]) and same_floats(g["coeff_ransac"], base["coeff_ransac"])
        assert_bit_equal(g["ground"][0], base["ground"][0], "ground")


def test_unknown_model_is_refused(cm):
    x = A.wall_zone(seed=62)
    for bad in (3, -1):
        with pytest.raises(Exception) as e:
            cm.plane_ransac(x, 0.3, model=bad)
        assert getattr(e.value, "code", None) == 1
        with pytest.raises(Exception) as e:
            cm.proceed_zones(x, [(20.0, -10.0, 2.0)], model=bad)
        assert getattr(e.value, "code", None) == 1


REAR_PARTS = ((30.0, 30.0, 2.0), (26.0, 4.0, 1.5), (8.0, -4.0, 0.3), (11.0, -15.0, 0.5))
TOP_PARTS = ((40.0, 20.0, 1.0), (35.0, -15.0, None))
LIVOX_PARTS = ((26.0, 34.0, 1.5), (10.0, 24.0, 1.2), (10.0, 14.0, 0.8), (10.0, 4.0, 0.5))


def oracle_proceed(oracle, roi, parts, p: NodeParams, model, eps):
    no_ground, ground, planes = [], [], []
    f32 = np.float32
    for (length, dev, zg) in parts:
        x = (0, float(f32(dev)), float(f32(f32(dev) + f32(length))), 0)
        part = np.ascontiguousarray(roi[oracle.passthrough(roi, *x[:3], False)])
        if zg is None:
            no_ground.append(part)
            continue
        low = np.ascontiguousarray(part[oracle.passthrough(part, 2, float(-f32(zg)), float(f32(zg)))])
        high = part[oracle.passthrough(part, 2, float(f32(np.float64(f32(zg)) + 0.01)), float(f32(p.roi_z_max)))]
        r = PO.plane_ransac_model(low, p.distance_threshold, p.prob, p.max_iterations, True, 12345, p.sum_order, model,
                                      A.Z, eps)
        rest = np.ascontiguousarray(np.delete(low, r["inliers"], axis=0))
        keep = oracle.radius_outlier(rest, p.radius, p.min_neighbor)
        no_ground += [rest[keep], high]
        ground.append(low[r["inliers"]])
        planes.append(r)
    cat = lambda xs: np.concatenate(xs) if xs else np.zeros((0, 4), np.float32)
    return cat(no_ground), cat(ground), planes


@pytest.mark.parametrize("name,parts", [("front", FRONT_PARTS), ("rear", REAR_PARTS), ("top", TOP_PARTS), ("livox", LIVOX_PARTS)])
@pytest.mark.parametrize("model", [A.PERP, A.PAR])
def test_proceed_zones_at_ten_degrees(gpu_ok, oracle, name, parts, model):
    """cm_proceed_zones / cm_dev_proceed_zones with the axis models at 10 degrees against the oracle's composition of
    getCloudPart + removeGround, for the reference's four zone tables."""
    p = NodeParams()
    mats = [synth.extrinsic(s, 2) for s in range(2)]
    with CloudMerger(max_sensors=1, max_points_per_sensor=1 << 17, max_batch_points=1 << 17, max_batch_frames=8) as cm:
        raw = synth.lidar_cloud(7300, 0, 0, 64, 1024)
        cur = oracle.transform(raw, mats[0][:3].reshape(-1))
        for (axis, lo, hi, neg) in p.roi_passes:
            cur = np.ascontiguousarray(cur[oracle.passthrough(cur, axis, lo, hi, bool(neg))])
        kw = dict(model=model, axis=A.Z, eps_angle=A.TEN_DEG)
        got = cm.proceed_zones(cur, parts, p.roi_z_max, p.radius, p.min_neighbor, p.distance_threshold, p.prob, p.max_iterations,
                               **kw)
        ng, g, planes = oracle_proceed(oracle, cur, parts, p, model, A.TEN_DEG)
        assert_bit_equal(got["no_ground"], ng, "%s no_ground" % name)
        assert_bit_equal(got["ground"], g, "%s ground" % name)
        assert len(got["planes"]) == len(planes)
        for a, b in zip(got["planes"], planes):
            for key in ("found", "iterations", "draws", "best_count", "rejected"):
                assert a[key] == b[key], (name, key)
            assert a["n_inliers"] == len(b["inliers"])
            assert same_floats(a["coeff"], b["coeff"]) and same_floats(a["coeff_ransac"], b["coeff_ransac"])
        buf = cm.upload(cur)
        dev = cm.dev_proceed_zones(buf.ptr, len(cur), parts, p.roi_z_max, p.radius, p.min_neighbor, p.distance_threshold, p.prob,
                                   p.max_iterations, **kw)
        assert dev["n_no_ground"] == len(ng) and dev["n_ground"] == len(g)
        assert_bit_equal(cm.download(dev["ground_ptr"], np.float32, 4 * len(g)).reshape(-1, 4), g, "%s device ground" % name)
        buf.free()
