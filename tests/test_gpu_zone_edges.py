"""GPU parity (-m gpu) of the zone slicing at its edges (tests/zone_edges.py, family Z): warp-row and tile edges,
16 zones over clouds past one and two rounds of k_zone_scan's tile loop, the box and chain membership paths on the same
windows, the regrowth of the outputs, and a zone total of 2^32 and more, which must be refused as CM_E_CAPACITY."""
import numpy as np
import pytest

import zone_edges as Z
from cloud_merger_b200 import CloudMerger, CloudMergerError, _lib
from helpers import assert_bit_equal

pytestmark = pytest.mark.gpu

CAP = 1 << 16


@pytest.fixture(scope="module")
def cm(gpu_ok):
    with CloudMerger(max_sensors=1, max_points_per_sensor=CAP, max_batch_points=CAP) as m:
        yield m


def _check(got, x, masks, what):
    assert len(got) == len(masks), what
    for k, ((gx, gi), m) in enumerate(zip(got, masks)):
        want = np.nonzero(m)[0]
        assert len(gi) == len(want) and (gi.astype(np.int64) == want).all(), "zone %d of %s" % (k, what)
        assert_bit_equal(gx, x[want], "zone %d coordinates of %s" % (k, what))


def split_both(cm, x, zones, what, host=True):
    """Device form (with its launch count) and host form; returns the device form's zones."""
    cm.set_zones(zones)
    buf = cm.upload(x) if len(x) else None
    cm.dev_zone_split(buf.ptr if buf else 0, len(x))
    assert cm.launch_count() == (3 if len(x) else 1), what
    got = cm.zone_out()
    if buf:
        buf.free()
    if host:
        h = cm.zone_split(x, capacity=max(len(zones) * len(x), 1))
        for (ax, ai), (bx, bi) in zip(got, h):
            assert np.array_equal(ai, bi) and ax.tobytes() == bx.tobytes(), what + " (host form)"
    return got


def test_zone_tile_edges(cm, oracle):
    for case in Z.tile_cases():
        x, zones = case["x"], case["zones"]
        masks = Z.np_zone_masks(x, zones)
        got = split_both(cm, x, zones, case["name"])
        _check(got, x, masks, case["name"])
        for k, (ox, oi) in enumerate(oracle.zone_split(x, zones)):
            assert np.array_equal(got[k][1], oi), (case["name"], k)


def test_zone_box_and_chain_paths_agree(cm, oracle):
    """Every window set as boxes (where derive_box allows it) and forced onto the chain path by the no-op stage: both
    equal oracle.zone_split and each other."""
    for case in Z.path_cases():
        x, zones = case["x"], case["zones"]
        want = oracle.zone_split(x, zones)
        masks = Z.np_zone_masks(x, zones)
        a = split_both(cm, x, zones, case["name"] + " (as given)")
        b = split_both(cm, x, Z.with_noop(zones), case["name"] + " (chain)")
        for k in range(len(zones)):
            assert np.array_equal(a[k][1], want[k][1]) and np.array_equal(b[k][1], want[k][1]), (case["name"], k)
            assert a[k][0].tobytes() == b[k][0].tobytes() == want[k][0].tobytes(), (case["name"], k)
        _check(a, x, masks, case["name"])


def test_zone_scan_rounds(cm):
    """16 zones with points in every round of k_zone_scan's 8192-tile loop (the s_run carry), box and chain path."""
    for n in Z.SCAN_NS:
        x = Z.scan_cloud(n)
        masks = Z.np_zone_masks(x, Z.SCAN_ZONES)
        for zones, what in ((Z.SCAN_ZONES, "box"), (Z.with_noop(Z.SCAN_ZONES), "chain")):
            got = split_both(cm, x, zones, "Z-scan %d %s" % (n, what), host=False)
            _check(got, x, masks, "Z-scan %d %s" % (n, what))


def test_zone_outputs_regrow(gpu_ok):
    """16 keep-all zones hold 16 n points, more than the outputs sized for 2 n (the handle's batch size is one tile):
    cm_get_zone_out grows them and repeats the scatter, which cm_launch_count then reports (3 launches before the
    fetch, 4 after)."""
    with CloudMerger(max_sensors=1, max_points_per_sensor=Z.ZN_TILE, max_batch_points=Z.ZN_TILE) as cm:
        _regrow(cm)


def _regrow(cm):
    for n in Z.GROW_NS:
        x = Z.scan_cloud(n, 5)
        cm.set_zones(Z.KEEP_ALL)
        buf = cm.upload(x)
        cm.dev_zone_split(buf.ptr, n)
        assert cm.launch_count() == 3
        got = cm.zone_out()
        assert cm.launch_count() == 4
        buf.free()
        for k, (gx, gi) in enumerate(got):
            assert len(gi) == n and (gi == np.arange(n, dtype=np.uint32)).all(), (n, k)
            assert_bit_equal(gx, x, "keep-all zone %d of %d points" % (k, n))


@pytest.mark.parametrize("n", [1 << 28, (1 << 28) + 64])
def test_zone_total_past_2_pow_32_is_refused(gpu_ok, n):
    """16 keep-all zones over 2^28 points hold 2^32 points together: the total must not wrap to a small number (the
    scatter would then write past the outputs); the split is refused as CM_E_CAPACITY and the handle stays usable."""
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < 20e9:
        pytest.skip("needs about 15 GB of free device memory")
    small = Z.scan_cloud(3000, 9)
    with CloudMerger(max_sensors=1, max_points_per_sensor=CAP, max_batch_points=CAP) as m:
        pts = torch.zeros((n, 4), dtype=torch.float32, device="cuda")
        m.set_zones(Z.KEEP_ALL)
        torch.cuda.synchronize()
        m.dev_zone_split(pts.data_ptr(), n)
        torch.cuda.synchronize()
        with pytest.raises(CloudMergerError) as e:
            m.zone_out()
        assert e.value.code == _lib.CM_E_CAPACITY, str(e.value)
        del pts
        torch.cuda.empty_cache()
        zones = Z.SCAN_ZONES
        got = split_both(m, small, zones, "after the refused split")
        _check(got, small, Z.np_zone_masks(small, zones), "after the refused split")
