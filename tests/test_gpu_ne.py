"""GPU parity tests (-m gpu) of the normal estimation (pcl::NormalEstimation with a radius search, PCL 1.8.1) through the
C ABI against the C++ statement of PCL's loop (tests/ne_oracle.cpp, the shared trig rule). Every case runs through the
four entry points (normals_multi, normals cloud by cloud, and their device forms), with the cell table and with the
binary searches (CM_NE_NO_TABLE). Bar: bit-exact normals and curvatures (NaN positions and bits included), the NaN counts,
the largest neighbourhood and the queries of each path, and cm_launch_count equal to the plan of the call. The struct
layout check against a compiled C program needs no GPU."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from cloud_merger_b200 import CloudMerger, CloudMergerError, _lib

import edge_inputs as E
import ne_cases as K
import ne_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
gpu = pytest.mark.gpu
WARP_CAP, CTA_CAP = _lib.CM_NE_WARP_CAP, _lib.CM_NE_CTA_CAP


def ne_launches(clouds, radius, table):
    """the radius removal's front end without its count kernel, then the gather, the warp and the CTA kernels"""
    plan = E.ror_plan(clouds, radius, table=table)
    n = sum(len(c) for c in clouds)
    return E.ror_launches(plan, clouds) - 1 + (3 if n else 0)


def _bits_equal(got, want, what):
    g, w = np.ascontiguousarray(got, F32).view(np.uint32), np.ascontiguousarray(want, F32).view(np.uint32)
    assert g.shape == w.shape, what
    bad = np.nonzero((g != w).any(axis=1))[0]
    assert len(bad) == 0, "%s: %d points differ, first %d: got %s want %s" % (
        what, len(bad), bad[0], got[bad[0]].tolist(), want[bad[0]].tolist())


def _device(cm, clouds, radius, vp, begin, single=False):
    allpts = np.ascontiguousarray(np.concatenate(clouds)) if begin[-1] else np.zeros((1, 4), F32)
    buf = cm.upload(allpts)
    try:
        if single:
            cm.dev_normals(buf.ptr, int(begin[-1]), radius, vp)
        else:
            cm.dev_normals_multi(buf.ptr, begin, radius, vp)
        return cm.normals_out()
    finally:
        buf.free()


def check(cm, monkeypatch, clouds, radius, vp=(0.0, 0.0, 0.0), tables=(True, False), singles=True):
    clouds = [np.ascontiguousarray(c, F32).reshape(-1, 4) for c in clouds]
    det = [O.normals(c, radius, vp, details=True) for c in clouds]
    want = [d[0] for d in det]
    counts = np.concatenate([d[1] for d in det]) if clouds else np.zeros(0)
    finite = np.concatenate([np.isfinite(c[:, :3]).all(axis=1) for c in clouds])
    stats = {"n_warp": int((finite & (counts <= WARP_CAP)).sum()),
             "n_cta": int((finite & (counts > WARP_CAP) & (counts <= CTA_CAP)).sum()),
             "n_multi": int((finite & (counts > CTA_CAP)).sum()),
             "max_neighbors": int(counts.max()) if len(counts) else 0,
             "n_nan": [int(np.isnan(w[:, 0]).sum()) for w in want]}
    begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    for table in tables:
        if table:
            monkeypatch.delenv("CM_NE_NO_TABLE", raising=False)
        else:
            monkeypatch.setenv("CM_NE_NO_TABLE", "1")
        what = "radius %r vp %r table %s" % (radius, vp, table)
        got = cm.normals_multi(clouds, radius, vp)
        for c, (g, w) in enumerate(zip(got, want)):
            _bits_equal(g, w, what + " (multi, cloud %d)" % c)
        assert cm.launch_count() == ne_launches(clouds, radius, table), what + " launches"
        out = _device(cm, clouds, radius, vp, begin)
        for c, w in enumerate(want):
            _bits_equal(out["normals"][begin[c]:begin[c + 1]], w, what + " (device multi, cloud %d)" % c)
        assert cm.launch_count() == ne_launches(clouds, radius, table), what + " launches (device)"
        for k, v in stats.items():
            assert out[k] == v, "%s: %s %r vs %r" % (what, k, out[k], v)
        assert out["host_syncs"] == 1
        if not singles:
            continue
        for c, (cloud, w) in enumerate(zip(clouds, want)):
            _bits_equal(cm.normals(cloud, radius, vp), w, what + " (single %d)" % c)
            if len(cloud):
                o = _device(cm, [cloud], radius, vp, np.array([0, len(cloud)], np.int64), single=True)
                _bits_equal(o["normals"], w, what + " (device single %d)" % c)
    return want, stats


@pytest.fixture(scope="module")
def cm(gpu_ok):
    with CloudMerger(max_sensors=1, max_points_per_sensor=1 << 21, max_batch_points=1 << 22, max_batch_frames=16) as m:
        yield m


@pytest.fixture(scope="module")
def roi58():
    return K.roi_cloud(7, 64, 2048)


@gpu
@pytest.mark.parametrize("radius", [0.1, 0.3, 0.5])
def test_roi_58k(cm, monkeypatch, roi58, radius):
    _, st = check(cm, monkeypatch, [roi58], radius, (0.0, 0.0, 1.8))
    assert st["n_warp"] > 0


@gpu
@pytest.mark.parametrize("radius", [0.1, 0.3, 0.5])
def test_roi_233k(cm, monkeypatch, radius):
    roi = K.roi_cloud(7, 128, 4096)
    _, st = check(cm, monkeypatch, [roi], radius)
    if radius == 0.5:
        assert st["n_cta"] > 0


@gpu
def test_zone_clouds_of_233k(cm, monkeypatch):
    check(cm, monkeypatch, K.zone_clouds(K.roi_cloud(7, 128, 4096)), 0.3)


@gpu
def test_fused_frame_2m(cm, monkeypatch):
    check(cm, monkeypatch, [K.fused_frame(3)], 0.1)


@gpu
@pytest.mark.parametrize("radius", [0.5, 0.1, 0.3, 1.0 / 3.0])
def test_ulp_edges_of_the_strict_bound(cm, monkeypatch, radius):
    c = K.ulp_edges(int(radius * 1000), radius)
    check(cm, monkeypatch, [c], radius, (1.0, 2.0, 3.0))


@gpu
@pytest.mark.parametrize("radius", [0.5, 0.1, 0.25])
def test_neighbours_across_cell_faces(cm, monkeypatch, radius):
    cell = float(F32(radius) * F32(1.00390625))
    check(cm, monkeypatch, [K.shell_faces(11, cell)], radius)


@gpu
def test_duplicates_lattice_ties_and_eigen_branches(cm, monkeypatch):
    lat = K.lattice(10, 0.25)
    check(cm, monkeypatch, [lat], 0.25)                                   # every lattice step exactly at r2: own point only
    check(cm, monkeypatch, [lat], float(np.nextafter(F32(0.25), F32(1))))
    check(cm, monkeypatch, [lat], 0.3)                                    # 6 ties at one distance: the index order decides
    check(cm, monkeypatch, [K.with_duplicates(lat, 5, 0.5), K.with_duplicates(K.blobs(6, 2000), 6, 0.5)], 0.4)
    check(cm, monkeypatch, [K.eigen_family(1, 0.3), K.small_groups(0.3)], 0.3, (0.5, -0.5, 2.0))


@gpu
@pytest.mark.parametrize("cap", [WARP_CAP, CTA_CAP])
def test_neighbourhoods_at_each_path_capacity(cm, monkeypatch, cap):
    _, st = check(cm, monkeypatch, [K.exact_neighbourhoods([cap - 1, cap, cap + 1], 0.3, seed=cap)], 0.3,
                  tables=(True, False))
    assert st["max_neighbors"] == cap + 1


@gpu
def test_dense_blob_on_the_multi_walk_path(cm, monkeypatch):
    _, st = check(cm, monkeypatch, [K.dense_blob(3, 20000, 0.3)], 0.3)
    assert st["n_multi"] == 20000


@gpu
def test_tiny_nonfinite_and_empty_clouds(cm, monkeypatch):
    a = K.with_nonfinite(K.blobs(13, 1500), 13, 0.1)
    nan_only = np.full((3, 4), np.nan, F32)
    empty = np.zeros((0, 4), F32)
    check(cm, monkeypatch, [a, K.small_groups(0.3), nan_only, empty], 0.3)
    check(cm, monkeypatch, [empty], 0.3)


@gpu
@pytest.mark.parametrize("vp", [(np.nan, 0.0, 0.0), (np.inf, 0.0, 0.0), (0.0, -np.inf, 1.0), "on_a_point"])
def test_viewpoints(cm, monkeypatch, vp):
    c = K.blobs(21, 3000)
    if vp == "on_a_point":
        vp = tuple(float(v) for v in c[17, :3])  # cos = +-0 at that point: no flip
    check(cm, monkeypatch, [c], 0.5, vp)


@gpu
def test_flip_decided_left_to_right(cm, monkeypatch):
    """viewpoints near a point's tangent plane where the order of the flip's dot product decides the flip"""
    for c, vp in K.flip_ties(5):
        check(cm, monkeypatch, [c], 1.0, vp)


@gpu
def test_sixteen_clouds_overlapping_and_empty(cm, monkeypatch):
    clouds = [K.blobs(100 + k, 300 + 97 * k) for k in range(14)]
    clouds[3] = np.zeros((0, 4), F32)
    clouds[9] = np.zeros((0, 4), F32)
    clouds.append(clouds[5].copy())  # the same space as cloud 5: no neighbours across clouds
    clouds.append(K.blobs(105, 800))
    check(cm, monkeypatch, clouds, 0.4, (0.0, 0.0, 10.0))


@gpu
def test_the_cell_bound(cm, monkeypatch):
    """|x| / cell just below 2^14 is served; just above it is CM_E_KEY_RANGE"""
    c = K.blobs(12, 3000, spread=1.0, outliers=0)
    cell = float(F32(0.5) * F32(1.00390625))
    inside = c.copy()
    inside[:, 0] = (inside[:, 0] - inside[:, 0].max() + F32(16383.5 * cell)).astype(F32)
    check(cm, monkeypatch, [inside], 0.5, tables=(True,))
    past = c.copy()
    past[:, 0] = (past[:, 0] - past[:, 0].min() + F32(16384.5 * cell)).astype(F32)
    for form in ("host", "device"):
        with pytest.raises(CloudMergerError) as e:
            if form == "host":
                cm.normals(past, 0.5)
            else:
                buf = cm.upload(past)
                try:
                    cm.dev_normals(buf.ptr, len(past), 0.5)
                    cm.normals_out()
                finally:
                    buf.free()
        assert e.value.code == _lib.CM_E_KEY_RANGE
    check(cm, monkeypatch, [inside], 0.5, tables=(True,))  # the handle is not affected


@gpu
def test_handle_reuse_after_radius_sor_and_cluster_calls(cm, monkeypatch, roi58):
    cm.radius_outlier(roi58, 0.15, 1)
    check(cm, monkeypatch, [roi58], 0.3)
    cm.statistical_outlier(roi58, 10, 1.0)
    check(cm, monkeypatch, K.zone_clouds(roi58, 3), 0.3)
    cm.euclidean_clusters(roi58, 0.5, 10, 25000)
    check(cm, monkeypatch, [roi58], 0.2)
    kx, ki = cm.radius_outlier(roi58, 0.15, 1)
    assert len(ki) > 0


@gpu
def test_refusals(cm, roi58):
    for bad in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(CloudMergerError) as e:
            cm.normals(roi58[:100], bad)
        assert e.value.code == _lib.CM_E_INVALID, bad
    with pytest.raises(CloudMergerError) as e:
        cm.normals_multi([roi58[:10]] * 17, 0.3)
    assert e.value.code == _lib.CM_E_INVALID


@gpu
def test_profiled_times(cm, roi58):
    cm.set_profiling(True)
    try:
        cm.normals(roi58, 0.5)
        out = cm.normals_out()
    finally:
        cm.set_profiling(False)
    assert out["warp_ms"] > 0 and out["cta_ms"] >= 0


def test_struct_sizes_match_a_compiled_c_program():
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "cloud_merger_gpu.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %d %d\n", sizeof(cm_ne_cfg_t), offsetof(cm_ne_cfg_t, viewpoint),
         offsetof(cm_ne_cfg_t, reserved), sizeof(cm_normal_out_t), offsetof(cm_normal_out_t, n_nan),
         offsetof(cm_normal_out_t, max_neighbors), offsetof(cm_normal_out_t, n_multi), offsetof(cm_normal_out_t, n_clouds),
         offsetof(cm_normal_out_t, host_syncs), offsetof(cm_normal_out_t, cta_ms), CM_NE_WARP_CAP, CM_NE_CTA_CAP);
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
    N = _lib.CmNormalOut
    want = [C.sizeof(_lib.CmNeCfg), _lib.CmNeCfg.viewpoint.offset, _lib.CmNeCfg.reserved.offset, C.sizeof(N),
            N.n_nan.offset, N.max_neighbors.offset, N.n_multi.offset, N.n_clouds.offset, N.host_syncs.offset,
            N.cta_ms.offset, WARP_CAP, CTA_CAP]
    assert got == want
