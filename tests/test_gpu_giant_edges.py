"""GPU parity of the giant-cloud mode at its edges (-m gpu): the edge clouds of tests/edge_inputs.py (key-width grids,
histogram-bin boundaries, lattices, kilometre offsets, signed zeros and subnormals, the key-range limits, degenerate clouds,
each with and without non-finite rows) through cm_giant_voxelgrid at world 1 (the product path), through its dry routing
for 2 to 16 virtual ranks, through the composition of the dry parts, and through the routing building blocks -- against the
independent numpy plan of tests/giant_reference.py and the float oracle."""
import numpy as np
import pytest

import edge_inputs as E
import giant_reference as R
from cloud_merger_b200 import CloudMerger, CloudMergerError, GiantCloud, _lib
from helpers import assert_bit_equal, assert_centroids_within_bound

pytestmark = pytest.mark.gpu

F32 = np.float32
WORLDS = (2, 3, 4, 8, 16)
NF = ["", "+nf"]


def _upload(cm, x):
    """A device copy of x (one dummy row for an empty cloud: the pointer must be valid, n is 0)."""
    return cm.upload(x if len(x) else np.zeros((1, 4), F32))


def _voxels(cm):
    st = cm.stats()
    v = int(st.voxels_out)
    o = cm.device_out()
    return (st, cm.download(o.voxel_idx, np.uint64, v).astype(np.int64), cm.download(o.voxel_count, np.uint32, v),
            cm.download(o.voxel_xyzi, F32, v * 4).reshape(v, 4))


def _check_oracle(x, leaf, min_points, idx, cnt, cen, oracle, what):
    o = oracle.voxelgrid(x, [leaf] * 3, min_points, True, force64=True, is_dense=False)
    assert len(idx) == o["n"], "%s: %d voxels vs oracle %d" % (what, len(idx), o["n"])
    assert (idx == o["idx"]).all() and (cnt == o["count"]).all(), "%s: voxel ids / counts / order differ" % what
    assert_bit_equal(cen, o["centroid"], "%s centroids vs float oracle" % what)
    assert_centroids_within_bound(cen, o["centroid_f64"], x, o["point_idx"], o["idx"], o["count"], what)
    return o


@pytest.mark.parametrize("nf", NF)
@pytest.mark.parametrize("case", E.GIANT_CASES)
def test_world1_product_path(gpu_ok, oracle, case, nf):
    """GiantCloud(cm, 0, 1): the grid, key width and finite count of the plan equal the reference; the local VoxelGrid sorts
    index bits (+1 for the sentinel frame of non-finite points) in ceil(bits / 8) passes without a device error, and its
    voxels equal the oracle's bit for bit, at min_points 1 and 2."""
    x, leaf = E.giant_case(case + nf)
    ref = R.grid(x, leaf)
    n = len(x)
    has_nf = bool((~R.finite_rows(x)).any())
    with CloudMerger(max_batch_points=max(n, 1)) as cm:
        buf = _upload(cm, x)
        g = GiantCloud(cm, 0, 1)
        try:
            for min_points in (1, 2):
                what = "%s%s min_points %d" % (case, nf, min_points)
                cm.set_voxel(leaf, min_points, True)
                info = g.voxelgrid(buf.ptr, n)
                st, idx, cnt, cen = _voxels(cm)
                fi = cm.frame_info()[0]
                assert info["min_b"].tolist() == ref["min_b"].tolist() and info["div_b"].tolist() == ref["div_b"].tolist(), what
                assert info["key_bits"] == ref["key_bits"], what
                assert info["points_total_finite"] == ref["finite"], what
                assert info["points_received"] == n and info["points_sent_away"] == 0
                assert st.device_error == 0, what
                if n:
                    bits = ref["key_bits"] + (1 if has_nf else 0)
                    assert st.key_bits == bits, (what, st.key_bits, bits)
                    assert st.sort_passes == max(1, -(-bits // 8)), what
                    assert st.key_bytes == (4 if bits <= 32 else 8), what
                o = _check_oracle(x, leaf, min_points, idx, cnt, cen, oracle, what)
                if ref["finite"]:
                    assert bool(fi.pcl_overflow) == bool(o["pcl_overflow"]), what
                else:
                    assert len(idx) == 0
        finally:
            g.close()


@pytest.mark.parametrize("case", E.GIANT_RANGE_CASES)
def test_world1_key_range_then_recovery(gpu_ok, oracle, case):
    """A cell origin at +-2^30 or 2^21 + 1 cells on an axis: cm_giant_voxelgrid itself refuses the plan with CM_E_KEY_RANGE in
    both overflow modes (with and without non-finite rows), in world 1 and in a dry routing; the same GiantCloud then gives
    oracle-exact voxels for a good cloud."""
    good, gleaf = E.giant_case("A:0.1+nf")
    clouds = [E.giant_case(case)[0], E.giant_case(case + "+nf")[0]]
    n = max(len(good), *(len(c) for c in clouds))
    with CloudMerger(max_batch_points=n) as cm:
        g = GiantCloud(cm, 0, 1)
        dry = GiantCloud(cm, 1, 4, None)
        try:
            for x in clouds:
                buf = _upload(cm, x)
                for pcl_like in (False, True):
                    cm.set_overflow_mode(pcl_like)
                    cm.set_voxel(1.0, 1, True)
                    for gc in (g, dry):
                        with pytest.raises(CloudMergerError) as e:
                            gc.voxelgrid(buf.ptr, len(x))
                        assert e.value.code == _lib.CM_E_KEY_RANGE, (case, pcl_like)
                buf.free()
            cm.set_overflow_mode(False)
            cm.set_voxel(gleaf, 1, True)
            buf = cm.upload(good)
            info = g.voxelgrid(buf.ptr, len(good))
            st, idx, cnt, cen = _voxels(cm)
            assert st.device_error == 0 and info["points_total_finite"] == R.grid(good, gleaf)["finite"]
            _check_oracle(good, gleaf, 1, idx, cnt, cen, oracle, "good cloud after %s" % case)
        finally:
            dry.close()
            g.close()


def _check_parts(got, x, p, W, me, what):
    """The grouping of a dry run against the reference plan: membership and source order, coordinates bit for bit, and the
    invariant itself -- every finite point of part r has a key in [s_{r-1}, s_r), every non-finite one is in part `me`."""
    assert len(got) == W, what
    split = [0] + list(p["splitters"])
    for r in range(W):
        xyzi, src = got[r]
        want = p["parts"][r]
        assert len(src) == len(want) and (src.astype(np.int64) == want).all(), "%s part %d: members / order" % (what, r)
        assert (xyzi.view(np.uint32) == x[want].view(np.uint32)).all(), "%s part %d: coordinates" % (what, r)
        k = p["keys"][src.astype(np.int64)]
        fin = k >= 0
        kf = k[fin].astype(np.uint64)
        inside = (kf >= np.uint64(split[r])) & ((kf < np.uint64(split[r + 1])) if r + 1 < W else True)
        assert np.all(inside), "%s part %d: a key outside its range" % (what, r)
        assert r == me or fin.all(), "%s: non-finite points left rank %d" % (what, me)


@pytest.mark.parametrize("nf", NF)
@pytest.mark.parametrize("case", E.GIANT_CASES)
def test_dry_routing(gpu_ok, case, nf):
    """GiantCloud(cm, me, W, None) on the whole cloud for W in 2..16 and me in {0, middle, W-1}: grid, splitters,
    send_begin, points_sent_away and points_total_finite equal the reference, and so does the grouping."""
    x, leaf = E.giant_case(case + nf)
    n = len(x)
    with CloudMerger(max_batch_points=max(n, 1)) as cm:
        cm.set_voxel(leaf, 1, True)
        buf = _upload(cm, x)
        for W in WORLDS:
            for me in sorted({0, W // 2, W - 1}):
                what = "%s%s W=%d me=%d" % (case, nf, W, me)
                p = R.plan(x, leaf, W, me)
                g = GiantCloud(cm, me, W, None)
                try:
                    info = g.voxelgrid(buf.ptr, n)
                    got = cm.zone_out()
                finally:
                    g.close()
                assert info["min_b"].tolist() == p["min_b"].tolist() and info["div_b"].tolist() == p["div_b"].tolist(), what
                assert info["key_bits"] == p["key_bits"], what
                assert info["splitters"] == p["splitters"], (what, info["splitters"], p["splitters"])
                assert info["points_total_finite"] == p["total"] == p["finite"], what
                assert info["send_begin"] == p["send_begin"], what
                assert info["points_sent_away"] == p["points_sent_away"], what
                _check_parts(got, x, p, W, me, what)


def test_seventeen_ranks_are_refused(gpu_ok):
    with CloudMerger(max_batch_points=16) as cm:
        with pytest.raises(CloudMergerError) as e:
            GiantCloud(cm, 0, 17, None)
        assert e.value.code == _lib.CM_E_INVALID


COMPOSE_CASES = ["bits:%d" % b for b in (8, 16, 24, 32, 33, 40)] + ["bin:w63", "bin:w2p40", "A:0.1", "A:0.035", "C:0.05",
                                                                    "Z:0.05", "origin:ok-", "axis:2p21", "deg:hot-voxel"]


@pytest.mark.parametrize("nf", NF)
@pytest.mark.parametrize("case", COMPOSE_CASES)
def test_dry_parts_compose_to_the_whole_cloud(gpu_ok, oracle, case, nf):
    """Every dry part through cm_set_voxel_bounds(global box) + cm_dev_voxelgrid: concatenated in rank order the voxels are
    the oracle's on the whole cloud -- no voxel straddles two ranks, also where rounding decides the cell."""
    x, leaf = E.giant_case(case + nf)
    n = len(x)
    for W, me in ((3, 1), (4, 3)):
        with CloudMerger(max_batch_points=n) as cm:
            cm.set_voxel(leaf, 1, True)
            buf = cm.upload(x)
            g = GiantCloud(cm, me, W, None)
            try:
                info = g.voxelgrid(buf.ptr, n)
                parts = cm.zone_out()
            finally:
                g.close()
        idx, cnt, cen = [], [], []
        with CloudMerger(max_batch_points=n) as cm:
            cm.set_voxel(leaf, 1, True)
            cm.set_voxel_bounds(info["min_p"], info["max_p"])
            for xyzi, _ in parts:
                if not len(xyzi):
                    continue
                b = cm.upload(np.ascontiguousarray(xyzi))
                cm.dev_voxelgrid(b.ptr, len(xyzi), False)
                st, i, c, z = _voxels(cm)
                assert st.device_error == 0
                idx.append(i); cnt.append(c); cen.append(z)
                b.free()
        _check_oracle(x, leaf, 1, np.concatenate(idx), np.concatenate(cnt), np.concatenate(cen), oracle,
                      "%s%s composed over W=%d" % (case, nf, W))


BLOCK_CASES = ["A:0.1", "A:0.035", "C:0.05", "bin:w1", "bin:w64", "bin:w63", "bin:w2p40", "bits:56"]


@pytest.mark.parametrize("nf", NF)
@pytest.mark.parametrize("case", BLOCK_CASES)
def test_key_histogram_and_route_by_key(gpu_ok, case, nf):
    """cm_dev_key_histogram at 4096 and 16384 bins (privatised in shared memory) and 65536 (global atomics), and
    cm_dev_route_by_key with the reference splitters, against the reference."""
    x, leaf = E.giant_case(case + nf)
    n = len(x)
    ref = R.grid(x, leaf)
    k = R.keys(x, leaf, ref["min_b"], ref["div_b"])
    with CloudMerger(max_batch_points=n) as cm:
        cm.set_voxel(leaf, 1, True)
        buf = cm.upload(x)
        for bins in (4096, 1 << 14, 1 << 16):
            hb = cm.device_buffer(bins * 8)
            width = cm.dev_key_histogram(buf.ptr, n, ref["min_p"], ref["max_p"], bins, hb.ptr)
            hist = cm.download(hb.ptr, np.uint64, bins).astype(np.int64)
            assert width == R.bin_width(ref["cells"], bins), (case, bins)
            want = R.histogram(k, ref["cells"], bins)
            assert (hist == want).all(), "%s%s bins %d: %d bins differ" % (case, nf, bins, int((hist != want).sum()))
            hb.free()
        for W, me in ((5, 2), (16, 0)):
            p = R.plan(x, leaf, W, me)
            cm.dev_route_by_key(buf.ptr, n, ref["min_p"], ref["max_p"], p["splitters"], me)
            _check_parts(cm.zone_out(), x, p, W, me, "%s%s route_by_key W=%d" % (case, nf, W))
