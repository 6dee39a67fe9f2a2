"""GPU parity tests (-m gpu) of the Euclidean cluster extraction (pcl::EuclideanClusterExtraction of PCL 1.8.1) through the
C ABI against the C++ statement of PCL's loop (tests/ec_oracle.cpp). Every case runs through the four entry points
(euclidean_clusters_multi, euclidean_clusters cloud by cloud, and their device forms), with the cell table and with the
binary searches (CM_EC_NO_TABLE). Bar: bit-exact cluster count, cluster order, indices and coordinates, and
cm_launch_count equal to the plan of the call. The struct-size check against a compiled C program needs no GPU."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from cloud_merger_b200 import CloudMerger, CloudMergerError, _lib

import ec_cases as K
import ec_oracle as O
import edge_inputs as E
from helpers import assert_bit_equal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
gpu = pytest.mark.gpu


def ec_launches(clouds, tolerance, table, n_clusters):
    """cm_launch_count of a call: the radius removal's front end without its count kernel; gather + hook, label + roots,
    the compaction of the kept roots; with kept clusters their sizes, ranks + keys, 3 per radix pass, the gather."""
    plan = E.ror_plan(clouds, float(F32(tolerance)), table=table)
    n = sum(len(c) for c in clouds)
    out = E.ror_launches(plan, clouds) - 1 + (4 if n else 0) + (3 if n else 1)
    if n_clusters:
        out += 1 + 2 + 3 * max(1, -(-n_clusters.bit_length() // 8)) + 1
    return out


def _same(got, want, clouds, what):
    assert len(got) == len(clouds), what
    for c, (g, w, cloud) in enumerate(zip(got, want, clouds)):
        assert len(g) == len(w), "%s: cloud %d: %d clusters vs %d" % (what, c, len(g), len(w))
        for j, ((gx, gi), wi) in enumerate(zip(g, w)):
            assert len(gi) == len(wi) and (gi.astype(np.int64) == wi).all(), "%s: cloud %d cluster %d" % (what, c, j)
            assert_bit_equal(gx, cloud[wi], "%s: cloud %d cluster %d coordinates" % (what, c, j))


def _device(cm, clouds, args, begin, single_cloud=None):
    allpts = np.ascontiguousarray(np.concatenate(clouds)) if begin[-1] else np.zeros((1, 4), F32)
    buf = cm.upload(allpts)
    try:
        if single_cloud is None:
            cm.dev_euclidean_clusters_multi(buf.ptr, begin, *args)
        else:
            cm.dev_euclidean_clusters(buf.ptr, int(begin[-1]), *args)
        out = cm.euclidean_clusters_out()
    finally:
        buf.free()
    got = []
    for c, cl in enumerate(out["clusters"]):
        res = []
        for ids in cl:
            res.append((allpts[ids.astype(np.int64)] if len(ids) else np.zeros((0, 4), F32),
                        (ids.astype(np.int64) - begin[c]).astype(np.uint32)))
        got.append(res)
    # the coordinates the call gathered, in output order
    flat = np.concatenate([i for cl in out["clusters"] for i in cl]).astype(np.int64) if len(out["xyzi"]) else None
    if flat is not None:
        assert_bit_equal(out["xyzi"], allpts[flat], "device xyzi")
    return got, out


def check(cm, monkeypatch, clouds, tolerance, min_size=1, max_size=O.INT_MAX, tables=(True, False)):
    clouds = [np.ascontiguousarray(c, F32).reshape(-1, 4) for c in clouds]
    want = [O.euclidean_clusters(c, tolerance, min_size, max_size) for c in clouds]
    begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    args = (tolerance, min_size, max_size)
    n_clusters = sum(len(w) for w in want)
    for table in tables:
        if table:
            monkeypatch.delenv("CM_EC_NO_TABLE", raising=False)
        else:
            monkeypatch.setenv("CM_EC_NO_TABLE", "1")
        what = "tol %r min %d max %d table %s" % (tolerance, min_size, max_size, table)
        _same(cm.euclidean_clusters_multi(clouds, *args, with_xyzi=True), want, clouds, what + " (multi)")
        assert cm.launch_count() == ec_launches(clouds, tolerance, table, n_clusters), what + " launches"
        got, out = _device(cm, clouds, args, begin)
        _same(got, want, clouds, what + " (device multi)")
        assert out["n_unclustered"] == begin[-1] - sum(len(i) for w in want for i in w)
        assert cm.launch_count() == ec_launches(clouds, tolerance, table, n_clusters), what + " launches (device)"
        for c, (cloud, w) in enumerate(zip(clouds, want)):
            _same([cm.euclidean_clusters(cloud, *args, with_xyzi=True)], [w], [cloud], what + " (single %d)" % c)
            if len(cloud):
                got, _ = _device(cm, [cloud], args, np.array([0, len(cloud)], np.int64), single_cloud=True)
                _same(got, [w], [cloud], what + " (device single %d)" % c)
    return want


@pytest.fixture(scope="module")
def cm(gpu_ok):
    with CloudMerger(max_sensors=1, max_points_per_sensor=1 << 21, max_batch_points=1 << 21, max_batch_frames=16) as m:
        yield m


@pytest.fixture(scope="module")
def roi58():
    return K.roi_cloud(7, 64, 2048)


@gpu
@pytest.mark.parametrize("min_size,max_size", [(1, O.INT_MAX), (10, 25000)])
def test_roi_58k(cm, monkeypatch, roi58, min_size, max_size):
    want = check(cm, monkeypatch, [roi58], 0.5, min_size, max_size)
    assert len(want[0]) > 5


@gpu
def test_roi_233k_and_zone_clouds(cm, monkeypatch):
    roi = K.roi_cloud(7, 128, 4096)
    check(cm, monkeypatch, [roi], 0.5, 10, 25000, tables=(True,))
    check(cm, monkeypatch, K.zone_clouds(roi), 0.5, 10, 25000)


@gpu
def test_fused_frame_2m(cm, monkeypatch):
    check(cm, monkeypatch, [K.fused_frame(3)], 0.2, 10, 25000, tables=(True,))


@gpu
@pytest.mark.parametrize("tolerance", [0.5, 0.1, 0.3, 1.0 / 3.0])
def test_ulp_pairs_on_the_strict_bound(cm, monkeypatch, tolerance):
    """steps of sqrt(r2) +- 1..3 ulps: chains join or break on the strict <; 0.1 and 1/3 are not floats, so r2 is the
    double square of the narrowed tolerance, not the radius removal's (float)(radius * radius)"""
    c = K.ulp_pairs(int(tolerance * 1000), tolerance)
    want = check(cm, monkeypatch, [c], tolerance)
    assert 0 < len(want[0]) < len(c)


@gpu
@pytest.mark.parametrize("tolerance", [0.5, 0.1, 0.25])
def test_pairs_across_cell_faces(cm, monkeypatch, tolerance):
    cell = float(F32(tolerance) * F32(1.00390625))
    check(cm, monkeypatch, [K.shell_faces(11, cell)], tolerance)


@gpu
def test_duplicates_and_lattice_ties(cm, monkeypatch):
    lat = K.lattice(10, 0.5)
    check(cm, monkeypatch, [lat], 0.5)                                   # every step exactly at r2: all singletons
    check(cm, monkeypatch, [lat], float(np.nextafter(F32(0.5), F32(1))))  # one ulp more: one cluster
    check(cm, monkeypatch, [K.with_duplicates(lat, 5, 0.5), K.with_duplicates(K.blobs(6, 2000), 6, 0.5)], 0.3)
    check(cm, monkeypatch, [np.repeat(K.blobs(7, 50, outliers=0), 4, axis=0)], 0.05)


@gpu
def test_snaking_chains(cm, monkeypatch):
    check(cm, monkeypatch, [K.snake(3, 0.5), K.snake(4, 0.2)], 0.5)


@gpu
@pytest.mark.parametrize("n_clusters,size", [(20, 5), (40, 7), (1500, 3)])
def test_equal_size_clusters(cm, monkeypatch, n_clusters, size):
    """more than 16 (introsort's partitioning path) and more than 10^3 clusters of one size, mixed with a few others"""
    c = K.equal_clusters(n_clusters, n_clusters, size, 0.5, extra=(size + 1, size - 1, size, 2 * size))
    want = check(cm, monkeypatch, [c], 0.5, tables=(True,))
    assert len(want[0]) == n_clusters + 4


@gpu
def test_min_max_filters(cm, monkeypatch):
    c = K.equal_clusters(8, 10, 6, 0.5, extra=(5, 7, 3))
    for mn, mx in ((5, 7), (6, 6), (7, 7), (5, 5), (8, 100), (0, 2 ** 31 - 1), (0, 0), (7, 6), (2 ** 31 - 1, 2 ** 31 - 1)):
        check(cm, monkeypatch, [c], 0.5, mn, mx, tables=(True,))


@gpu
def test_nonfinite_empty_and_tiny_clouds(cm, monkeypatch):
    a = K.with_nonfinite(K.blobs(13, 1500), 13, 0.1)
    one = K.blobs(14, 1, outliers=0)
    two = np.array([[0, 0, 0, 1], [0.2, 0, 0, 2]], F32)
    nan_only = np.full((3, 4), np.nan, F32)
    empty = np.zeros((0, 4), F32)
    check(cm, monkeypatch, [a, one, two, nan_only, empty], 0.3)
    check(cm, monkeypatch, [empty], 0.3)
    check(cm, monkeypatch, [two], 0.1)


@gpu
def test_sixteen_clouds_overlapping_and_empty(cm, monkeypatch):
    clouds = [K.blobs(100 + k, 300 + 97 * k) for k in range(14)]
    clouds[3] = np.zeros((0, 4), F32)
    clouds[9] = np.zeros((0, 4), F32)
    clouds.append(clouds[5].copy())  # the same space as cloud 5: no cluster across clouds
    clouds.append(K.blobs(105, 800))
    check(cm, monkeypatch, clouds, 0.4, 3, 1000)


@gpu
def test_utm_offset_and_the_cell_bound(cm, monkeypatch):
    """|x| / cell just below 2^14 is served; just above it is CM_E_KEY_RANGE (from the call itself)"""
    c = K.blobs(12, 3000, spread=1.0, outliers=0)
    cell = float(F32(0.5) * F32(1.00390625))
    inside = c.copy()
    inside[:, 0] = (inside[:, 0] - inside[:, 0].max() + F32(16383.5 * cell)).astype(F32)
    check(cm, monkeypatch, [inside], 0.5, 5, 25000)
    far = K.roi_cloud(3, 32, 512) + np.array([5.0e5, 5.0e5, 0, 0], F32)
    check(cm, monkeypatch, [far], 40.0, tables=(True,))
    past = c.copy()
    past[:, 0] = (past[:, 0] - past[:, 0].min() + F32(16384.5 * cell)).astype(F32)
    for form in ("host", "device"):
        with pytest.raises(CloudMergerError) as e:
            if form == "host":
                cm.euclidean_clusters(past, 0.5)
            else:
                buf = cm.upload(past)
                try:
                    cm.dev_euclidean_clusters(buf.ptr, len(past), 0.5)
                finally:
                    buf.free()
        assert e.value.code == _lib.CM_E_KEY_RANGE
    check(cm, monkeypatch, [inside], 0.5, 5, 25000, tables=(True,))  # the handle is not affected


@gpu
def test_handle_reuse_after_radius_sor_and_zone_calls(cm, monkeypatch, roi58):
    radius = float(F32(0.15))
    cm.radius_outlier(roi58, radius, 1)
    check(cm, monkeypatch, [roi58], 0.5, 10, 25000, tables=(True,))
    cm.statistical_outlier(roi58, 10, 1.0)
    check(cm, monkeypatch, K.zone_clouds(roi58, 3), 0.5, 10, 25000, tables=(True,))
    cm.set_zones([[(0, -15.0, 20.0, 0)], [(0, 20.0, 60.0, 0)]])
    z = cm.zone_split(roi58)
    assert len(z[0][1]) + len(z[1][1]) == len(roi58)
    check(cm, monkeypatch, [roi58], 0.5, 10, 25000, tables=(True,))
    kx, ki = cm.radius_outlier(roi58, radius, 1)
    assert len(ki) > 0


@gpu
def test_capacity_and_refusals(cm, roi58):
    small = K.equal_clusters(1, 6, 4, 0.5)
    cfg = _lib.CmEcCfg(0.5, 1, 2 ** 31 - 1)
    n = len(small)
    ox, oi, cb = np.zeros((n, 4), F32), np.zeros(n, np.uint32), np.zeros(n + 1, np.int64)
    nc, npo = C.c_int64(), C.c_int64()
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    for pcap, ccap in ((n - 1, 6), (n, 5)):
        rc = cm._lib.cm_euclidean_clusters(cm._h, ptr(small), n, C.byref(cfg), ptr(ox), ptr(oi), pcap,
                                           cb.ctypes.data_as(C.POINTER(C.c_int64)), ccap, C.byref(nc), C.byref(npo))
        assert rc == _lib.CM_E_CAPACITY and nc.value == 6 and npo.value == n
    for bad in (dict(tolerance=0.0), dict(tolerance=-1.0), dict(tolerance=float("nan")), dict(tolerance=float("inf")),
                dict(tolerance=1e300), dict(tolerance=1e-50), dict(min_size=-1), dict(max_size=-1)):
        kw = dict(tolerance=0.5, min_size=1, max_size=100)
        kw.update(bad)
        with pytest.raises(CloudMergerError) as e:
            cm.euclidean_clusters(roi58[:100], **kw)
        assert e.value.code == _lib.CM_E_INVALID, bad


def test_struct_sizes_match_a_compiled_c_program():
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "cloud_merger_gpu.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(cm_ec_cfg_t), offsetof(cm_ec_cfg_t, max_size), sizeof(cm_cluster_out_t),
         offsetof(cm_cluster_out_t, n_clusters), offsetof(cm_cluster_out_t, cloud_clusters), offsetof(cm_cluster_out_t, n_clouds),
         offsetof(cm_cluster_out_t, host_syncs), offsetof(cm_cluster_out_t, hook_ms), offsetof(cm_cluster_out_t, reserved));
  return 0;
}
'''
    with tempfile.TemporaryDirectory() as d:
        with open(os.path.join(d, "s.c"), "w") as f:
            f.write(src)
        exe = os.path.join(d, "s")
        subprocess.run([os.environ.get("CC", "gcc"), "-I", os.path.join(ROOT, "include"), "-o", exe, os.path.join(d, "s.c")],
                       check=True)
        got = [int(v) for v in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    O_ = _lib.CmClusterOut
    want = [C.sizeof(_lib.CmEcCfg), _lib.CmEcCfg.max_size.offset, C.sizeof(O_), O_.n_clusters.offset,
            O_.cloud_clusters.offset, O_.n_clouds.offset, O_.host_syncs.offset, O_.hook_ms.offset, O_.reserved.offset]
    assert got == want
