"""GPU parity (-m gpu) of the radius outlier removal at its edges (tests/edge_inputs.py, family N): the cell margin up to
2^14 - 1 cells from the origin, the direct-address table's gaps and bounds, every key width and radix pass parity, the
count's early exit, and the refusals (CM_E_KEY_RANGE) of grids the plan cannot serve. Every case runs through the four
entry points, with the table and with the binary searches, keep and negative; survivors must be bit-exact against the C++
oracle per cloud. cm_get_stats does not describe a radius run (it has no centroid stage), so the plan that ran is checked
through cm_launch_count: a bounding box per cloud, grid setup, keys, one launch per radix pass (so the pass count and its
parity; 5 and 6 passes mean 64-bit keys), the table when it is used, the count."""
import numpy as np
import pytest

import edge_inputs as E
from cloud_merger_b200 import CloudMerger, CloudMergerError, _lib
from helpers import assert_bit_equal

pytestmark = pytest.mark.gpu

CASES = E.ror_cases()
REFUSED = E.ror_refused_cases()
CAP = 40000


@pytest.fixture(scope="module")
def cm(gpu_ok):
    with CloudMerger(max_sensors=1, max_points_per_sensor=CAP, max_batch_points=CAP, max_batch_frames=8) as m:
        yield m


def _check_multi(got, clouds, wants, what):
    assert len(got) == len(clouds)
    for c, (gx, gi), want in zip(clouds, got, wants):
        assert len(gi) == len(want) and (gi.astype(np.int64) == want).all(), what
        assert_bit_equal(gx, c[want], what)


@pytest.mark.parametrize("name", sorted(CASES))
def test_ror_edges_bit_exact(cm, oracle, monkeypatch, name):
    clouds, r, min_pts = CASES[name]
    begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    buf = cm.upload(np.ascontiguousarray(np.concatenate(clouds)))
    for table in (True, False):
        plan = E.ror_plan(clouds, r, table=table)
        if not table and not E.ror_plan(clouds, r)["table"]:
            continue                                   # the searches ran already
        if table:
            monkeypatch.delenv("CM_ROR_NO_TABLE", raising=False)
        else:
            monkeypatch.setenv("CM_ROR_NO_TABLE", "1")
        launches = E.ror_launches(plan, clouds)
        for m in min_pts:
            for neg in (False, True):
                what = "%s table=%s min_pts=%d negative=%s" % (name, table, m, neg)
                wants = [oracle.radius_outlier(c, r, m, neg).astype(np.int64) for c in clouds]
                _check_multi(cm.radius_outlier_multi(clouds, r, m, neg), clouds, wants, what + " (multi)")
                assert cm.launch_count() == launches, what
                cm.dev_radius_outlier_multi(buf.ptr, begin, r, m, neg)
                zones = cm.zone_out()
                _check_multi([(x, i.astype(np.int64) - begin[k]) for k, (x, i) in enumerate(zones)], clouds, wants,
                             what + " (device multi)")
                assert cm.launch_count() == launches, what
                if len(clouds) == 1:
                    gx, gi = cm.radius_outlier(clouds[0], r, m, neg)
                    _check_multi([(gx, gi)], clouds, wants, what + " (single)")
                    cm.dev_radius_outlier(buf.ptr, len(clouds[0]), r, m, neg)
                    _check_multi([cm.radius_outlier_out()], clouds, wants, what + " (device single)")
                    assert cm.launch_count() == launches, what
    monkeypatch.delenv("CM_ROR_NO_TABLE", raising=False)


def _refused(fn):
    with pytest.raises(CloudMergerError) as e:
        fn()
    assert e.value.code == _lib.CM_E_KEY_RANGE, str(e.value)


@pytest.mark.parametrize("name", sorted(REFUSED))
def test_ror_refusals(cm, oracle, monkeypatch, name):
    """Grids beyond the key range (N-range: refused before the table and the count) and clouds 2^14 cells from the origin
    (N-bound: refused by the count kernel, reported by cm_get_zone_out for the device forms) give CM_E_KEY_RANGE from every
    entry point, and the next call on the handle succeeds."""
    clouds, r = REFUSED[name]
    begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    buf = cm.upload(np.ascontiguousarray(np.concatenate(clouds)))
    good = CASES["count:hot"][0][0]
    want = oracle.radius_outlier(good, r, 1, False)
    for table in (True, False):
        if table:
            monkeypatch.delenv("CM_ROR_NO_TABLE", raising=False)
        else:
            monkeypatch.setenv("CM_ROR_NO_TABLE", "1")
        _refused(lambda: cm.radius_outlier_multi(clouds, r, 1))
        if name.startswith("range:"):
            _refused(lambda: cm.dev_radius_outlier_multi(buf.ptr, begin, r, 1))
        else:
            cm.dev_radius_outlier_multi(buf.ptr, begin, r, 1)
            _refused(cm.zone_out)
        if len(clouds) == 1:
            _refused(lambda: cm.radius_outlier(clouds[0], r, 1))
            if name.startswith("range:"):
                _refused(lambda: cm.dev_radius_outlier(buf.ptr, len(clouds[0]), r, 1))
            else:
                cm.dev_radius_outlier(buf.ptr, len(clouds[0]), r, 1)
                _refused(cm.radius_outlier_out)
        gx, gi = cm.radius_outlier(good, r, 1)                  # the handle goes on
        assert (gi == want).all()
        assert_bit_equal(gx, good[want], "after a refusal")
    monkeypatch.delenv("CM_ROR_NO_TABLE", raising=False)


def test_proceed_zones_refuses_a_radius_too_small_for_the_roi(gpu_ok):
    """proceedX's outlier stage on a 60 m ROI at radius 1e-3 (2^14 cells are 16.4 m) is refused with CM_E_KEY_RANGE; the
    next pass on the handle at the usual radius succeeds."""
    rng = np.random.default_rng(8)
    n = 20000
    roi = np.column_stack([rng.uniform(0, 60, n), rng.uniform(-5, 5, n), rng.uniform(-1.9, 2.5, n),
                           rng.uniform(0, 255, n)]).astype(np.float32)
    roi[: n // 2, 2] = (-1.8 + rng.normal(0, 0.02, n // 2)).astype(np.float32)
    parts = [(30.0, 0.0, 2.0), (30.0, 30.0, 2.0)]
    with CloudMerger(max_sensors=1, max_points_per_sensor=n, max_batch_points=2 * n, max_batch_frames=4) as m:
        _refused(lambda: m.proceed_zones(roi, parts, radius=1e-3))
        out = m.proceed_zones(roi, parts, radius=0.15)
        assert len(out["no_ground"]) > 0 and len(out["ground"]) > 0


ZONE_CHUNK = 8192 * 1024      # points per chunk of k_zone_scan (8192 tiles of 1024)


@pytest.mark.parametrize("n", [ZONE_CHUNK - 1, ZONE_CHUNK + 1, 9_500_000])
def test_zone_split_across_scan_chunks(gpu_ok, n):
    """Zone slicing past one chunk of k_zone_scan: the running carry between chunks must reach every later tile."""
    rng = np.random.default_rng(n)
    x = np.column_stack([rng.uniform(-10, 70, n), rng.uniform(-5, 5, n), rng.uniform(-1, 3, n),
                         np.zeros(n)]).astype(np.float32)
    zones = [[(0, 0.0, 20.0, 0)], [(0, 15.0, 60.0, 0), (2, -0.5, 2.0, 0)], [(1, -1.0, 1.0, 1)]]
    masks = [(x[:, 0] >= 0) & (x[:, 0] <= 20),
             (x[:, 0] >= 15) & (x[:, 0] <= 60) & (x[:, 2] >= -0.5) & (x[:, 2] <= 2),
             (x[:, 1] < -1) | (x[:, 1] > 1)]
    with CloudMerger(max_sensors=1, max_points_per_sensor=n, max_batch_points=16) as m:
        m.set_zones(zones)
        got = m.zone_split(x)
    for (gx, gi), mk in zip(got, masks):
        want = np.nonzero(mk)[0]
        assert len(gi) == len(want) and (gi.astype(np.int64) == want).all()
        assert_bit_equal(gx, x[want], "zone points")


def test_ror_lattice_beyond_one_scan_chunk(gpu_ok):
    """About 9.5 M points of a 0.1 m lattice at radius 0.15 and min_pts 18: an interior point has exactly 19 points inside
    the radius (itself, 6 at 0.1 m, 12 at 0.141 m), a point on the lattice's surface fewer, so exactly the interior
    survives -- through the compaction's carry across chunks."""
    s = 212
    g = np.stack(np.meshgrid(np.arange(s), np.arange(s), np.arange(s), indexing="ij"), axis=-1).reshape(-1, 3)
    rng = np.random.default_rng(12)
    perm = rng.permutation(len(g))
    g = g[perm]
    x = np.column_stack([(g * 0.1).astype(np.float32), np.zeros(len(g), np.float32)]).astype(np.float32)
    interior = ((g > 0) & (g < s - 1)).all(axis=1)
    want = np.nonzero(interior)[0]
    assert len(x) > ZONE_CHUNK
    with CloudMerger(max_sensors=1, max_points_per_sensor=len(x), max_batch_points=len(x)) as m:
        gx, gi = m.radius_outlier(x, float(np.float32(0.15)), 18)
    assert len(gi) == len(want) and (gi.astype(np.int64) == want).all()
    assert_bit_equal(gx, x[want], "lattice survivors")
