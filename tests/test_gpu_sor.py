"""GPU parity tests (-m gpu) of the statistical outlier removal (pcl::StatisticalOutlierRemoval of PCL 1.8.1) through the C
ABI against the numpy restatement of tests/sor_np.py. Bar: bit-exact per-point mean distances, per-cloud mean / stddev /
threshold, survivor set, order and coordinates."""
import numpy as np
import pytest

from cloud_merger_b200 import CloudMerger, CloudMergerError, _lib

import sor_cases as K
import sor_np
from helpers import assert_bit_equal

pytestmark = pytest.mark.gpu


def _same(a, b):
    return (np.isnan(a) and np.isnan(b)) or np.float64(a).tobytes() == np.float64(b).tobytes()


def check(cm, clouds, mean_k, std_mul, negative=False, sqrt_mode=0, device=False):
    """runs the clouds in one call and compares everything with the restatement; returns the GPU's statistics."""
    want = sor_np.sor(clouds, mean_k, std_mul, negative, sqrt_mode)
    begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    if device:
        allpts = np.ascontiguousarray(np.concatenate(clouds)) if begin[-1] else np.zeros((1, 4), np.float32)
        buf = cm.upload(allpts)
        cm.dev_statistical_outlier_multi(buf.ptr, begin, mean_k, std_mul, negative, sqrt_mode)
        zones = cm.zone_out()
        got = [(x, (i.astype(np.int64) - begin[c]).astype(np.uint32)) for c, (x, i) in enumerate(zones)]
    else:
        got = cm.statistical_outlier_multi(clouds, mean_k, std_mul, negative, sqrt_mode)
    out = cm.statistical_outlier_out()
    assert len(out["clouds"]) == len(clouds)
    for c, (cloud, w, (gx, gi)) in enumerate(zip(clouds, want, got)):
        assert_bit_equal(out["distances"][begin[c]:begin[c + 1]], w["distances"], "distances of cloud %d" % c)
        st = out["clouds"][c]
        assert st["n_valid"] == w["n_valid"] and st["too_few"] == w["too_few"], (c, st, w["n_valid"])
        if not w["too_few"]:
            for k in ("mean", "stddev", "threshold"):
                assert _same(st[k], w[k]), (c, k, st[k], w[k])
        keep = np.nonzero(w["keep"])[0]
        assert len(gi) == len(keep) and (gi == keep).all(), "survivor set / order of cloud %d" % c
        assert_bit_equal(gx, cloud[keep], "survivor coordinates of cloud %d" % c)
    return out


@pytest.fixture(scope="module")
def cm(gpu_ok):
    with CloudMerger(max_sensors=1, max_points_per_sensor=1 << 21, max_batch_points=1 << 21, max_batch_frames=16) as m:
        yield m


@pytest.fixture(scope="module")
def roi58():
    return K.roi_cloud(7, 64, 2048)


@pytest.mark.parametrize("mean_k", [1, 10, 50, 127])
@pytest.mark.parametrize("sqrt_mode", [0, 1])
def test_roi_cloud(cm, roi58, mean_k, sqrt_mode):
    out = check(cm, [roi58], mean_k, 1.0, sqrt_mode=sqrt_mode)
    assert not out["clouds"][0]["too_few"]


@pytest.mark.parametrize("std_mul,negative", [(0.0, False), (-0.5, False), (2.0, False), (1.0, True), (0.0, True)])
def test_std_mul_and_negative(cm, std_mul, negative):
    check(cm, [K.blobs(3, 3000)], 8, std_mul, negative)


@pytest.mark.parametrize("mean_k", [1, 50, 127])
def test_exactly_mean_k_plus_one_finite_points(cm, mean_k):
    c = np.concatenate([K.blobs(mean_k, mean_k + 1, outliers=0), np.full((2, 4), np.nan, np.float32)])
    out = check(cm, [c], mean_k, 1.0)
    assert not out["clouds"][0]["too_few"] and out["clouds"][0]["n_valid"] == mean_k + 1


def test_duplicates_and_lattice_ties(cm):
    lat = K.lattice(12)
    check(cm, [lat, K.with_duplicates(lat, 5, 0.5), K.with_duplicates(K.blobs(6, 2000), 6)], 6, 1.0)
    check(cm, [lat], 18, 1.0)  # 6 + 12 neighbours: the k-th value is tied with 11 others


def test_all_equal_distances_give_a_nan_threshold(cm):
    """every distance equal (a lattice, mean_k 1): with a step whose float square rounds down, sq_sum falls below
    sum * sum / valid, the variance is slightly negative and the NaN threshold keeps every point in both modes."""
    step = next(s for s in np.linspace(0.1, 0.3, 200, dtype=np.float32)
                if np.isnan(sor_np.sor_cloud(K.lattice(6, float(s)), 1, 1.0)["threshold"]))
    lat = K.lattice(6, float(step))
    for negative in (False, True):
        out = check(cm, [lat], 1, 1.0, negative)
        assert np.isnan(out["clouds"][0]["threshold"])
    check(cm, [np.concatenate([lat, lat])], 1, 1.0, True)  # all distances 0: threshold 0, negative removes everything


@pytest.mark.parametrize("cell", ["0.05", "0.3", "1000"])
def test_cell_edges_and_shell_faces(cm, monkeypatch, cell):
    """neighbours on grid faces and one or two ulps off them, under tiny, ordinary and one-cell grids"""
    monkeypatch.setenv("CM_SOR_CELL", cell)
    check(cm, [K.shell_faces(11, float(np.float32(0.3)))], 12, 1.0)


@pytest.mark.parametrize("cell", [None, "1000"])
def test_far_outliers(cm, monkeypatch, cell):
    """outliers hundreds of metres out: the search around them grows through many empty cubes"""
    if cell:
        monkeypatch.setenv("CM_SOR_CELL", cell)
    check(cm, [K.blobs(9, 4000, spread=0.3, outliers=40, far=200.0)], 10, 1.0)


def test_tiny_cells(cm, monkeypatch):
    """cells far below the neighbour distances: every search runs through several growth steps"""
    monkeypatch.setenv("CM_SOR_CELL", "0.01")
    check(cm, [K.blobs(10, 3000, spread=0.3, outliers=0)], 10, 1.0)


def test_utm_offset(cm):
    c = K.blobs(12, 5000, spread=2.0, outliers=10)
    off = c.copy()
    off[:, 0] = (off[:, 0] + np.float32(5.0e5)).astype(np.float32)
    off[:, 1] = (off[:, 1] - np.float32(4.2e6)).astype(np.float32)
    check(cm, [off], 10, 1.0)
    check(cm, [K.roi_cloud(3, 32, 512) + np.array([5.0e5, 5.0e5, 0, 0], np.float32)], 20, 1.0)


def test_nonfinite_rows_and_too_few(cm):
    a = K.with_nonfinite(K.blobs(13, 1500), 13, 0.1)
    few = K.with_nonfinite(K.blobs(14, 6, outliers=0), 14, 0.3)
    nan_only = np.full((4, 4), np.nan, np.float32)
    out = check(cm, [a, few, nan_only], 10, 1.0)
    assert out["clouds"][1]["too_few"] and not out["clouds"][0]["too_few"] and not out["clouds"][2]["too_few"]
    assert out["clouds"][2]["n_valid"] == 0
    out = check(cm, [a, few], 10, 1.0, negative=True)
    assert out["clouds"][1]["too_few"]


def test_sixteen_clouds_overlapping_and_empty(cm):
    clouds = [K.blobs(100 + k, 300 + 97 * k) for k in range(14)]
    clouds[3] = np.zeros((0, 4), np.float32)
    clouds[9] = np.zeros((0, 4), np.float32)
    clouds.append(clouds[5].copy())  # the same space as cloud 5: no neighbours across clouds
    clouds.append(K.blobs(105, 800))
    assert len(clouds) == 16
    check(cm, clouds, 7, 1.5)
    check(cm, clouds, 7, 1.5, device=True)


def test_sum_paths(cm, monkeypatch):
    """a cloud whose values fail the exactness condition (values spread over many binades with low set bits) takes the
    serial chain; an ordinary one the parallel sum; the hook forces the chain for both, with the same bits."""
    rng = np.random.default_rng(21)
    wide = np.concatenate([K.blobs(21, 2000, spread=1e-3), K.blobs(22, 2000, spread=3e3)])
    wide[:, :3] += rng.uniform(-1e-3, 1e-3, (len(wide), 3)).astype(np.float32)
    small = K.lattice(6, step=0.5)
    out = check(cm, [wide, small], 5, 1.0)
    paths = [c["sum_path"] for c in out["clouds"]]
    assert paths[1] == 0, paths
    assert paths[0] & _lib.CM_SOR_SQ_SUM_SERIAL, paths
    monkeypatch.setenv("CM_SOR_SERIAL_SUMS", "1")
    out = check(cm, [wide, small], 5, 1.0)
    assert all(c["sum_path"] == 3 for c in out["clouds"])


@pytest.mark.parametrize("table", [True, False])
def test_table_and_binary_search_lookups(cm, monkeypatch, roi58, table):
    if not table:
        monkeypatch.setenv("CM_SOR_NO_TABLE", "1")
    check(cm, K.zone_clouds(roi58), 10, 1.0, device=True)


def test_roi_233k(cm):
    check(cm, [K.roi_cloud(7, 128, 4096)], 50, 1.0)


def test_fused_frame_2m(cm):
    check(cm, [K.fused_frame(3)], 10, 1.0, device=True)


def test_handle_reuse_after_radius_and_zone_calls(cm, roi58):
    radius = float(np.float32(0.15))
    cm.radius_outlier(roi58, radius, 1)
    check(cm, [roi58], 10, 1.0)
    cm.set_zones([[(0, -15.0, 20.0, 0)], [(0, 20.0, 60.0, 0)]])
    cm.zone_split(roi58)
    check(cm, K.zone_clouds(roi58, 3), 10, 1.0, device=True)
    kx, ki = cm.radius_outlier(roi58, radius, 1)
    assert len(ki) > 0


def test_refusals(cm, roi58):
    for bad in (dict(mean_k=0), dict(mean_k=128), dict(std_mul=float("nan")), dict(sqrt_mode=2)):
        kw = dict(mean_k=10, std_mul=1.0, sqrt_mode=0)
        kw.update(bad)
        with pytest.raises(CloudMergerError) as e:
            cm.statistical_outlier(roi58[:100], **kw)
        assert e.value.code == _lib.CM_E_INVALID
    # the survivors of the previous call live in the zone outputs: they cannot be the input of the next one
    buf = cm.upload(roi58)
    cm.dev_statistical_outlier(buf.ptr, len(roi58), 10, 1.0)
    zo = _lib.CmZoneOut()
    assert cm._lib.cm_get_zone_out(cm._h, zo) == _lib.CM_OK
    with pytest.raises(CloudMergerError) as e:
        cm.dev_statistical_outlier(zo.xyzi, int(zo.begin[1]), 10, 1.0)
    assert e.value.code == _lib.CM_E_INVALID
