"""GPU parity tests (-m gpu) of the RANSAC ground plane (the pcl::SACSegmentation + pcl::ExtractIndices block of
removeGround(), pc_preprocessing_main.cpp:95-117; Parameter.h:38-42) through the C ABI against the oracle's restatement of
PCL 1.8.1 (sampler, model, stopping rule, least-squares refit). Bar: the same draw stream, model, iteration count and
inlier set as PCL's sequential loop -- bit-exact coefficients, indices and coordinates."""
import numpy as np
import pytest

from cloud_merger_b200 import CloudMerger

from helpers import assert_bit_equal, same_floats

pytestmark = pytest.mark.gpu

THR = float(np.float32(0.3))     # `const float distance_threshold = 0.3;` widened to setDistanceThreshold's double
PROB = float(np.float32(0.99))   # `const float prob = 0.99;`


def ground_scene(seed, n, ground_frac=0.7, slope=0.02, noise=0.03):
    rng = np.random.default_rng(seed)
    g = int(n * ground_frac)
    pts = np.zeros((n, 4), np.float32)
    pts[:, 0] = rng.uniform(-30, 30, n)
    pts[:, 1] = rng.uniform(-10, 10, n)
    pts[:g, 2] = -1.8 + slope * pts[:g, 0] + rng.normal(0, noise, g)
    pts[g:, 2] = rng.uniform(-1.5, 1.0, n - g)
    pts[:, 3] = rng.uniform(0, 255, n)
    return pts[rng.permutation(n)]


def check(cm, oracle, cloud, thr=THR, prob=PROB, max_it=1000, optimize=True, seed=12345, order=0, device_form=False):
    want = oracle.plane_ransac(cloud, thr, prob, max_it, optimize, seed, order)
    if device_form:
        buf = cm.upload(cloud)
        got = cm.dev_plane_ransac(buf.ptr, len(cloud), thr, prob, max_it, optimize, seed, order)
        zones = cm.zone_out()
        got["ground"], got["rest"] = zones[0], zones[1]
    else:
        got = cm.plane_ransac(cloud, thr, prob, max_it, optimize, seed, order)
    for key in ("found", "iterations", "draws", "best_count"):
        assert got[key] == want[key], (key, got[key], want[key])
    assert (got["sample"] == want["sample"]).all()
    assert same_floats(got["coeff_ransac"], want["coeff_ransac"]), (got["coeff_ransac"], want["coeff_ransac"])
    assert same_floats(got["coeff"], want["coeff"]), (got["coeff"], want["coeff"])
    gx, gi = got["ground"]
    rx, ri = got["rest"]
    assert got["n_inliers"] == len(want["inliers"]) == len(gi)
    assert (gi == want["inliers"]).all(), "inlier set / order differs"
    rest = np.setdiff1d(np.arange(len(cloud)), want["inliers"])
    assert len(ri) == len(rest) and (ri == rest).all(), "ExtractIndices(negative) set / order differs"
    assert_bit_equal(gx, cloud[want["inliers"]], "ground coordinates")
    assert_bit_equal(rx, cloud[rest], "no-ground coordinates")
    return want


@pytest.mark.parametrize("order", [0, 1, 2])
@pytest.mark.parametrize("optimize", [False, True])
def test_plane_ransac_matches_oracle(gpu_ok, oracle, order, optimize):
    with CloudMerger(max_sensors=1, max_points_per_sensor=60000, max_batch_points=60000) as cm:
        for seed, n, frac in ((1, 50000, 0.8), (2, 20000, 0.45), (3, 777, 0.7), (4, 5, 1.0), (5, 4, 1.0), (6, 3, 1.0)):
            w = check(cm, oracle, ground_scene(seed, n, frac), optimize=optimize, order=order)
            assert w["found"]
        check(cm, oracle, ground_scene(7, 30000, 0.8), optimize=optimize, order=order, device_form=True)


def test_plane_ransac_long_runs_and_caps(gpu_ok, oracle):
    """More hypotheses than one batch holds (the stopping rule needs several hundred iterations), the iteration cap, other
    seeds, a threshold that is not a float."""
    with CloudMerger(max_sensors=1, max_points_per_sensor=40000, max_batch_points=40000) as cm:
        weak = ground_scene(11, 30000, 0.12)
        w = check(cm, oracle, weak, prob=0.999999)
        assert w["iterations"] > 300
        w = check(cm, oracle, weak, prob=0.999999999, max_it=1500)
        assert w["iterations"] > 1024
        w = check(cm, oracle, weak, prob=0.999999, max_it=100)
        assert w["iterations"] == 101
        rng = np.random.default_rng(5)
        blob = rng.uniform(-20, 20, (20000, 4)).astype(np.float32)
        w = check(cm, oracle, blob, thr=0.05, max_it=1000)
        assert w["iterations"] == 1001
        for seed in (1, 99, 2**31 + 7):
            check(cm, oracle, ground_scene(12, 10000, 0.6), seed=seed)
        check(cm, oracle, ground_scene(13, 10000, 0.6), thr=0.3)   # the double 0.3, not 0.3f
        check(cm, oracle, ground_scene(13, 10000, 0.6), thr=0.0)   # nothing is strictly inside 0
        check(cm, oracle, ground_scene(14, 10000, 0.6, noise=0.0), thr=1e-6)


def test_plane_ransac_degenerate_inputs(gpu_ok, oracle):
    """Fewer than three points, collinear clouds (every draw rejected, getSamples gives up after 1000), duplicate points,
    non-finite points (never inliers; they stay in the no-ground cloud as ExtractIndices(negative) leaves them)."""
    with CloudMerger(max_sensors=1, max_points_per_sensor=4096, max_batch_points=4096) as cm:
        for n in (0, 1, 2):
            w = check(cm, oracle, ground_scene(20, 8, 1.0)[:n])
            assert not w["found"]
        t = np.arange(50, dtype=np.float32)
        line = np.column_stack([t, 2 * t, 4 * t, t]).astype(np.float32)
        w = check(cm, oracle, line)
        assert not w["found"] and w["draws"] == 1000
        dup = np.repeat(ground_scene(21, 40, 1.0), 5, axis=0)   # coincident sample points: zero normal, Eigen 3.3 normalize
        check(cm, oracle, dup)
        check(cm, oracle, np.repeat(np.array([[1, 2, 3, 4]], np.float32), 30, axis=0))
        bad = ground_scene(22, 3000, 0.8)
        bad[::97, 0] = np.nan
        bad[5::131, 2] = np.inf
        check(cm, oracle, bad)
        with pytest.raises(Exception):
            cm.plane_ransac(bad, THR, sum_order=7)


def test_plane_ransac_multi_equals_separate_searches(gpu_ok, oracle):
    """Five ground zones of one sensor cloud in one call (what a proceedX of the reference runs one after the other,
    pc_preprocessing_main.cpp:228-312) -- every cloud must come out exactly as its own search: different sizes, one empty,
    one below three points, one collinear, one that needs several batches."""
    t = np.arange(40, dtype=np.float32)
    clouds = [ground_scene(31, 20000, 0.8), ground_scene(32, 3000, 0.5), np.zeros((0, 4), np.float32),
              ground_scene(33, 9000, 0.12), ground_scene(34, 2, 1.0), np.column_stack([t, 2 * t, 4 * t, t]).astype(np.float32),
              ground_scene(35, 12345, 0.65), ground_scene(36, 513, 0.9)]
    begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    allpts = np.ascontiguousarray(np.concatenate(clouds))
    with CloudMerger(max_sensors=1, max_points_per_sensor=len(allpts), max_batch_points=len(allpts)) as cm:
        buf = cm.upload(allpts)
        for prob, optimize, order in ((PROB, True, 0), (0.999999, True, 1), (PROB, False, 2)):
            got = cm.dev_plane_ransac_multi(buf.ptr, begin, THR, prob, 1000, optimize, 12345, order)
            zones = cm.zone_out()
            assert len(zones) == 2 * len(clouds)
            for k, cloud in enumerate(clouds):
                want = oracle.plane_ransac(cloud, THR, prob, 1000, optimize, 12345, order)
                g = got[k]
                for key in ("found", "iterations", "draws", "best_count"):
                    assert g[key] == want[key], (k, key, g[key], want[key])
                assert (g["sample"] == want["sample"]).all()
                assert same_floats(g["coeff_ransac"], want["coeff_ransac"]) and same_floats(g["coeff"], want["coeff"])
                gx, gi = zones[2 * k]
                rx, ri = zones[2 * k + 1]
                assert g["n_inliers"] == len(want["inliers"]) == len(gi)
                assert (gi.astype(np.int64) - begin[k] == want["inliers"]).all()
                rest = np.setdiff1d(np.arange(len(cloud)), want["inliers"])
                assert (ri.astype(np.int64) - begin[k] == rest).all()
                assert_bit_equal(gx, cloud[want["inliers"]], "ground coordinates")
                assert_bit_equal(rx, cloud[rest], "no-ground coordinates")
        with pytest.raises(Exception):
            cm.dev_plane_ransac_multi(buf.ptr, np.arange(10, dtype=np.int64), THR)   # nine clouds


def test_plane_ransac_multi_host_form(gpu_ok, oracle):
    clouds = [ground_scene(41, 7000, 0.8), ground_scene(42, 100, 0.9), np.zeros((0, 4), np.float32), ground_scene(43, 2500, 0.4)]
    with CloudMerger(max_sensors=1, max_points_per_sensor=16384, max_batch_points=16384) as cm:
        got = cm.plane_ransac_multi(clouds, THR, PROB)
        for cloud, g in zip(clouds, got):
            want = oracle.plane_ransac(cloud, THR, PROB)
            assert (g["found"], g["iterations"], g["draws"]) == (want["found"], want["iterations"], want["draws"])
            assert same_floats(g["coeff"], want["coeff"])
            assert (g["ground"][1] == want["inliers"]).all()
            rest = np.setdiff1d(np.arange(len(cloud)), want["inliers"])
            assert (g["rest"][1] == rest).all()
            assert_bit_equal(g["ground"][0], cloud[want["inliers"]], "ground coordinates")
            assert_bit_equal(g["rest"][0], cloud[rest], "no-ground coordinates")


def test_plane_ransac_golden_fixture(gpu_ok):
    """The committed fixture tests/golden/plane_ransac.json (numpy restatement, no refit) through the C ABI."""
    import json
    import os
    doc = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "plane_ransac.json")))
    with CloudMerger(max_sensors=1, max_points_per_sensor=4096, max_batch_points=4096) as cm:
        for c in doc["cases"]:
            x = np.array(c["xyzi"], np.float32)
            e = c["expected"]
            r = cm.plane_ransac(x, c["threshold"], c["probability"], c["max_iterations"], False, c["seed"], c["sum_order"])
            assert (r["found"], r["iterations"], r["draws"], r["best_count"]) == (e["found"], e["iterations"], e["draws"], e["best_count"])
            assert r["sample"].tolist() == e["sample"]
            if e["found"]:
                assert r["coeff_ransac"].view(np.uint32).tolist() == e["coeff_ransac_bits"]
            assert r["ground"][1].tolist() == e["inliers"]


def test_stage_input_must_not_alias_the_handles_own_outputs(gpu_ok):
    """A stage writes into its handle's zone outputs; feeding it a cloud that lives there is refused, not corrupted."""
    from cloud_merger_b200 import CloudMergerError
    cloud = ground_scene(51, 4000, 0.8)
    with CloudMerger(max_sensors=1, max_points_per_sensor=8192, max_batch_points=8192) as cm:
        buf = cm.upload(cloud)
        cm.dev_plane_ransac(buf.ptr, len(cloud), THR)
        xyzi, _, begin = cm.zone_out_raw()
        for call in (lambda: cm.dev_plane_ransac(xyzi, begin[1], THR),
                     lambda: cm.dev_radius_outlier(xyzi + begin[1] * 16, begin[2] - begin[1], 0.15, 1),
                     lambda: (cm.set_zones([[(2, -1.0, 1.0, 0)]]), cm.dev_zone_split(xyzi, begin[1]))):
            with pytest.raises(CloudMergerError):
                call()
        # the same cloud through a second handle is fine
        with CloudMerger(max_sensors=1, max_points_per_sensor=8192, max_batch_points=8192) as other:
            r = other.dev_plane_ransac(xyzi, begin[1], THR)
            assert r["found"]
