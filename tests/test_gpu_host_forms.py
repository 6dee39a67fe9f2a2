"""GPU tests (-m gpu) of the copy-out of the host-buffer forms, called through the C ABI (the Python wrappers size their
outputs to fit). With a caller capacity one point short, every form returns CM_E_CAPACITY with the needed size in its last
offset (or n_out) and writes nothing past its arrays; with the capacity exact, it returns what the device form computes."""
import ctypes as C

import numpy as np
import pytest

from cloud_merger_b200 import CloudMerger, _lib

pytestmark = pytest.mark.gpu

GUARD_F, GUARD_I, GUARD_B = np.float32(-1234.5), np.uint32(0xA5A5A5A5), -77
RADIUS, MIN_NEIGHBORS = 0.3, 2
THR = 0.3


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _scene(seed, n):
    """A ground patch, clutter above it and a few far-off points: every filter keeps some points and drops others."""
    rng = np.random.default_rng(seed)
    pts = np.zeros((n, 4), np.float32)
    pts[:, 0] = rng.uniform(-10, 20, n)
    pts[:, 1] = rng.uniform(-3, 3, n)
    g = n * 2 // 3
    pts[:g, 2] = -1.8 + rng.normal(0, 0.03, g)
    pts[g:, 2] = rng.uniform(-1.5, 2.5, n - g)
    pts[:, 3] = rng.uniform(0, 255, n)
    far = rng.choice(n, n // 50, replace=False)
    pts[far, :3] += rng.uniform(-40, 40, (len(far), 3)).astype(np.float32)
    return pts


CLOUD = _scene(1, 3000)
CLOUDS = [_scene(2, 2500), _scene(3, 1500), _scene(4, 2000)]
PACKED = np.ascontiguousarray(np.concatenate(CLOUDS))
BEGIN = np.concatenate([[0], np.cumsum([len(c) for c in CLOUDS])]).astype(np.int64)


@pytest.fixture(scope="module")
def cm(gpu_ok):
    with CloudMerger(max_sensors=1, max_points_per_sensor=1 << 16, max_batch_points=1 << 16, max_batch_frames=16) as m:
        yield m


def _zones(cm):
    """The device form's result as one array with offsets, as the host forms return it."""
    zones = cm.zone_out()
    return (np.concatenate([x for x, _ in zones]), np.concatenate([i for _, i in zones]),
            np.concatenate([[0], np.cumsum([len(x) for x, _ in zones])]).astype(np.int64))


def _check_form(host, n_offsets, want):
    """host(capacity, out_xyzi, out_idx, out_begin) -> return code; want = the device form's (xyzi, idx, begin)."""
    want_x, want_i, want_b = want
    need = int(want_b[-1])
    assert len(want_b) == n_offsets and 0 < need
    for cap in (need - 1, need):
        ox = np.full((cap + 1, 4), GUARD_F, np.float32)   # one guard row / element behind the capacity
        oi = np.full(cap + 1, GUARD_I, np.uint32)
        ob = np.full(n_offsets + 1, GUARD_B, np.int64)
        rc = host(cap, ox, oi, ob)
        assert rc == (_lib.CM_OK if cap == need else _lib.CM_E_CAPACITY), (cap, need, rc)
        assert ob[:n_offsets].tolist() == want_b.tolist() and ob[n_offsets] == GUARD_B
        assert (ox[cap] == GUARD_F).all() and oi[cap] == GUARD_I
        if cap == need:
            assert ox[:need].tobytes() == want_x.tobytes() and (oi[:need] == want_i).all()


def _single(fn, *args):
    """A single-cloud form that reports n_out: its count as the offsets [0, n_out]."""
    def host(cap, ox, oi, ob):
        n_out = C.c_int64(-1)
        rc = fn(*args, _ptr(ox), _ptr(oi), C.c_int64(cap), C.byref(n_out))
        ob[0], ob[1] = 0, n_out.value
        return rc
    return host


def _offsets(ob):
    return ob.ctypes.data_as(C.POINTER(C.c_int64))


def test_zone_split_with_overlapping_zones(cm):
    zones = [[(0, -10.0, 8.0, 0)], [(0, 0.0, 20.0, 0)], [(2, -2.0, -1.6, 0), (1, -3.0, 3.0, 0)]]
    cm.set_zones(zones)
    cm.dev_zone_split(cm.upload(CLOUD).ptr, len(CLOUD))
    want = _zones(cm)
    assert want[2][-1] > len(CLOUD)   # the zones overlap

    def host(cap, ox, oi, ob):
        return cm._lib.cm_zone_split(cm._h, _ptr(CLOUD), len(CLOUD), _ptr(ox), _ptr(oi), cap, _offsets(ob))
    _check_form(host, len(zones) + 1, want)


def test_radius_outlier(cm):
    cm.dev_radius_outlier(cm.upload(CLOUD).ptr, len(CLOUD), RADIUS, MIN_NEIGHBORS)
    want = _zones(cm)
    assert 0 < want[2][-1] < len(CLOUD)
    _check_form(_single(cm._lib.cm_radius_outlier, cm._h, _ptr(CLOUD), len(CLOUD), RADIUS, MIN_NEIGHBORS, 0), 2, want)


def test_radius_outlier_multi(cm):
    cm.dev_radius_outlier_multi(cm.upload(PACKED).ptr, BEGIN, RADIUS, MIN_NEIGHBORS)
    want = _zones(cm)
    b = (C.c_int64 * len(BEGIN))(*BEGIN.tolist())

    def host(cap, ox, oi, ob):
        return cm._lib.cm_radius_outlier_multi(cm._h, _ptr(PACKED), b, len(CLOUDS), RADIUS, MIN_NEIGHBORS, 0, _ptr(ox),
                                               _ptr(oi), cap, _offsets(ob))
    _check_form(host, len(CLOUDS) + 1, want)


def test_statistical_outlier(cm):
    cfg = cm._sor_cfg(8, 1.0, False, 0)
    cm.dev_statistical_outlier(cm.upload(CLOUD).ptr, len(CLOUD), 8, 1.0)
    want = _zones(cm)
    assert 0 < want[2][-1] < len(CLOUD)
    _check_form(_single(cm._lib.cm_statistical_outlier, cm._h, _ptr(CLOUD), len(CLOUD), C.byref(cfg)), 2, want)


def test_statistical_outlier_multi(cm):
    cfg = cm._sor_cfg(8, 1.0, False, 0)
    cm.dev_statistical_outlier_multi(cm.upload(PACKED).ptr, BEGIN, 8, 1.0)
    want = _zones(cm)
    b = (C.c_int64 * len(BEGIN))(*BEGIN.tolist())

    def host(cap, ox, oi, ob):
        return cm._lib.cm_statistical_outlier_multi(cm._h, _ptr(PACKED), b, len(CLOUDS), C.byref(cfg), _ptr(ox), _ptr(oi),
                                                    cap, _offsets(ob))
    _check_form(host, len(CLOUDS) + 1, want)


def test_plane_ransac(cm):
    cfg = cm._plane_cfg(THR, 0.99, 1000, True, 12345, 0)
    cm.dev_plane_ransac(cm.upload(CLOUD).ptr, len(CLOUD), THR)
    want = _zones(cm)
    pl = _lib.CmPlane()

    def host(cap, ox, oi, ob):
        return cm._lib.cm_plane_ransac(cm._h, _ptr(CLOUD), len(CLOUD), C.byref(cfg), C.byref(pl), _ptr(ox), _ptr(oi), cap,
                                       _offsets(ob))
    _check_form(host, 3, want)


def test_plane_ransac_multi(cm):
    cfg = cm._plane_cfg(THR, 0.99, 1000, True, 12345, 0)
    cm.dev_plane_ransac_multi(cm.upload(PACKED).ptr, BEGIN, THR)
    want = _zones(cm)
    b = (C.c_int64 * len(BEGIN))(*BEGIN.tolist())
    pl = (_lib.CmPlane * len(CLOUDS))()

    def host(cap, ox, oi, ob):
        return cm._lib.cm_plane_ransac_multi(cm._h, _ptr(PACKED), b, len(CLOUDS), C.byref(cfg), pl, _ptr(ox), _ptr(oi), cap,
                                             _offsets(ob))
    _check_form(host, 2 * len(CLOUDS) + 1, want)


def test_proceed_zones(cm):
    """Two outputs with a capacity each: either one short refuses the call with both sizes reported."""
    parts = [(20.0, -10.0, 2.0), (12.0, 8.0, None)]
    args = (parts, 3.0, RADIUS, MIN_NEIGHBORS, THR, 0.99, 1000, True, 12345, 0)
    dev = cm.dev_proceed_zones(cm.upload(CLOUD).ptr, len(CLOUD), *args)
    n_ng, n_g = dev["n_no_ground"], dev["n_ground"]
    assert n_ng > 0 and n_g > 0
    want_ng = cm.download(dev["no_ground_ptr"], np.float32, 4 * n_ng).reshape(-1, 4)
    want_g = cm.download(dev["ground_ptr"], np.float32, 4 * n_g).reshape(-1, 4)
    cfg = cm._proceed_cfg(*args)
    pl = (_lib.CmPlane * _lib.CM_MAX_PROCEED_PARTS)()
    for cap_ng, cap_g in ((n_ng - 1, n_g), (n_ng, n_g - 1), (n_ng, n_g)):
        ng = np.full((cap_ng + 1, 4), GUARD_F, np.float32)
        g = np.full((cap_g + 1, 4), GUARD_F, np.float32)
        got_ng, got_g = C.c_int64(-1), C.c_int64(-1)
        rc = cm._lib.cm_proceed_zones(cm._h, _ptr(CLOUD), len(CLOUD), C.byref(cfg), _ptr(ng), cap_ng, C.byref(got_ng),
                                      _ptr(g), cap_g, C.byref(got_g), pl)
        fits = (cap_ng, cap_g) == (n_ng, n_g)
        assert rc == (_lib.CM_OK if fits else _lib.CM_E_CAPACITY), (cap_ng, cap_g, rc)
        assert (got_ng.value, got_g.value) == (n_ng, n_g)
        assert (ng[cap_ng] == GUARD_F).all() and (g[cap_g] == GUARD_F).all()
        if fits:
            assert ng[:n_ng].tobytes() == want_ng.tobytes() and g[:n_g].tobytes() == want_g.tobytes()
