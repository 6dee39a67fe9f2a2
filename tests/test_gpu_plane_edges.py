"""GPU parity (-m gpu) of the RANSAC ground plane at its edges (tests/plane_edges.py, family P): round edges, the
rejection limit, score chunks, moment tiles, the refit floor, thresholds, settings, eight-cloud layouts and clouds past
the compaction scan's rounds. Every case runs through plane_ransac, plane_ransac_multi, dev_plane_ransac and
dev_plane_ransac_multi; multi-cloud layouts also go cloud by cloud. Everything must be bit-exact against
cmo_plane_ransac, and cm_launch_count must equal plane_launches."""
import numpy as np
import pytest

import plane_edges as P
from cloud_merger_b200 import CloudMerger
from helpers import assert_bit_equal, same_floats

pytestmark = pytest.mark.gpu

CASES = P.plane_cases()
CAP = 1 << 16


@pytest.fixture(scope="module")
def cm(gpu_ok):
    with CloudMerger(max_sensors=1, max_points_per_sensor=CAP, max_batch_points=CAP) as m:
        yield m


def _check(got, ground, rest, cloud, want, optimize, what):
    for key in ("found", "iterations", "draws", "best_count"):
        assert got[key] == want[key], (what, key, got[key], want[key])
    assert (got["sample"] == want["sample"]).all(), what
    assert same_floats(got["coeff_ransac"], want["coeff_ransac"]), (what, got["coeff_ransac"], want["coeff_ransac"])
    assert same_floats(got["coeff"], want["coeff"]), (what, got["coeff"], want["coeff"])
    gx, gi = ground
    rx, ri = rest
    assert got["n_inliers"] == len(want["inliers"]) == len(gi), what
    if not optimize:   # without the refit, select keeps exactly the points the score kernel counted for the best draw
        assert got["best_count"] == got["n_inliers"], what
    assert (np.asarray(gi, np.int64) == want["inliers"]).all(), "inlier set / order of " + what
    others = np.setdiff1d(np.arange(len(cloud)), want["inliers"])
    assert len(ri) == len(others) and (np.asarray(ri, np.int64) == others).all(), "rest set / order of " + what
    assert_bit_equal(gx, cloud[want["inliers"]], "ground coordinates of " + what)
    assert_bit_equal(rx, cloud[others], "rest coordinates of " + what)


def run_four(cm, oracle, case, optimize, order):
    clouds = case["clouds"]
    args = (case["threshold"], case["probability"], case["max_iterations"], optimize, case["seed"], order)
    want = [oracle.plane_ransac(c, *args) for c in clouds]
    begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    n = int(begin[-1])
    launches = P.plane_launches([w["draws"] for w in want], optimize, any(w["found"] for w in want), n)
    what = "%s, optimize %d, order %d" % (case["name"], optimize, order)
    allpts = np.ascontiguousarray(np.concatenate(clouds))
    got = cm.plane_ransac_multi(clouds, *args)
    assert cm.launch_count() == launches, what + " (multi)"
    for k, (c, g, w) in enumerate(zip(clouds, got, want)):
        _check(g, g["ground"], g["rest"], c, w, optimize, "%s, cloud %d (multi)" % (what, k))
    buf = cm.upload(allpts) if n else None
    got = cm.dev_plane_ransac_multi(buf.ptr if buf else 0, begin, *args)
    assert cm.launch_count() == launches, what + " (device multi)"
    zones = cm.zone_out()
    for k, (c, g, w) in enumerate(zip(clouds, got, want)):
        gx, gi = zones[2 * k]
        rx, ri = zones[2 * k + 1]
        _check(g, (gx, gi.astype(np.int64) - begin[k]), (rx, ri.astype(np.int64) - begin[k]), c, w, optimize,
               "%s, cloud %d (device multi)" % (what, k))
    if buf:
        buf.free()
    for k, (c, w) in enumerate(zip(clouds, want)):   # cloud by cloud against the oracle's single search
        one = P.plane_launches([w["draws"]], optimize, w["found"], len(c))
        g = cm.plane_ransac(c, *args)
        assert cm.launch_count() == one, what + " (single)"
        _check(g, g["ground"], g["rest"], c, w, optimize, "%s, cloud %d (single)" % (what, k))
        if not len(c):
            continue
        b = cm.upload(c)
        g = cm.dev_plane_ransac(b.ptr, len(c), *args)
        assert cm.launch_count() == one, what + " (device single)"
        z = cm.zone_out()
        _check(g, z[0], z[1], c, w, optimize, "%s, cloud %d (device single)" % (what, k))
        b.free()


@pytest.mark.parametrize("family", ["P-batch", "P-bad", "P-chunk", "P-tile", "P-thr", "P-settings", "P-multi"])
def test_plane_edges_match_the_oracle(cm, oracle, family):
    for name, case in sorted(CASES.items()):
        if not name.startswith(family + ":"):
            continue
        for optimize in case["optimizes"]:
            for order in case["orders"]:
                run_four(cm, oracle, case, optimize, order)


def test_plane_edges_past_the_scan_rounds(gpu_ok, oracle):
    """A cloud of 8388609 points and eight clouds of 2 x 8388608 + 777: the given-mask compaction runs a second and a
    third round of k_zone_scan's tile loop."""
    with CloudMerger(max_sensors=1, max_points_per_sensor=CAP, max_batch_points=CAP) as m:
        for case in P.size_cases():
            run_four(m, oracle, case, True, 0)
