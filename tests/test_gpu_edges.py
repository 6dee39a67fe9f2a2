"""GPU parity at the rounding and grid-size edges (-m gpu): the inputs of tests/edge_inputs.py through every path that computes
a voxel key -- the dense VoxelGrid, K1's fused crop-box keys, the frame-segmented sort of a batch, the host path with its
captured and replayed graphs, global bounds -- against the float oracle (bit-exact) and against a float64 reference within
the derived bound of a float32 centroid (helpers.assert_centroids_within_bound)."""
import numpy as np
import pytest

import edge_inputs as E
from cloud_merger_b200 import CloudMerger, CloudMergerError, _lib, make_layout
from helpers import (assert_bit_equal, assert_centroids_within_bound, check_survivors, check_voxels, cloud_dict,
                     upload_segments)
from oracle import np_oracle

pytestmark = pytest.mark.gpu

PACKED = (16, 0, 4, 8, 12)
BOX_T = (1.25, 0.5, 0.375)
BOX = [(-2.5, 7.25), (-3.0, 3.5), (-1.5, 2.0)]
INT_WINDOW = (10.0, 200.0)


def _bound_check(out, frames_info, oracle_frames, points_of_frame):
    """Every frame's centroids against the float64 oracle within the derived float32 bound."""
    for f, (fi, o) in enumerate(zip(frames_info, oracle_frames)):
        v0, v1 = fi.voxel_begin, fi.voxel_end
        assert_centroids_within_bound(out["voxel_xyzi"][v0:v1], o["centroid_f64"], points_of_frame[f], o["point_idx"],
                                      o["idx"], o["count"], "frame %d" % f)


def _dense_case(name):
    """(cloud, leaf) of the dense-VoxelGrid cases."""
    kind, arg = name.split(":")
    if kind == "A":
        return E.lattice_cloud(300, float(arg), n_lattice=60000, n_filler=40000), float(arg)
    if kind == "C":
        return E.offset_cloud(301, float(arg), n=120000), float(arg)
    div = {"2p31": E.DIV_2P31, "2p31+": E.DIV_2P31_PLUS, "2p32": E.DIV_2P32, "2p32+": E.DIV_2P32_PLUS,
           "guard-": E.DIV_GUARD_BELOW, "guard+": E.DIV_GUARD_ABOVE, "axis2p21": (1 << 21, 3, 2)}
    if arg == "guard-disagrees":
        return E.grid_cloud(302, E.DIV_GUARD_ABOVE, n_filler=30000, inset=0.9), 1.0
    if arg.startswith("origin"):
        sign = -1.0 if arg.endswith("-") else 1.0
        return E.grid_cloud(303, (4, 5, 6), n_filler=5000, origin=(sign * E.ORIGIN_OK, 0.0, 0.0)), 1.0
    return E.grid_cloud(304, div[arg], n_filler=30000), 1.0


DENSE_CASES = (["A:%r" % leaf for leaf in E.LEAVES] + ["C:0.02", "C:0.05", "C:0.1"] +
               ["D:%s" % k for k in ("2p31", "2p31+", "2p32", "2p32+", "guard-", "guard+", "guard-disagrees", "axis2p21",
                                    "origin+", "origin-")])


@pytest.mark.parametrize("case", DENSE_CASES)
@pytest.mark.parametrize("is_dense", [1, 0])
def test_dense_voxelgrid_edges(gpu_ok, oracle, case, is_dense):
    """cm_dev_voxelgrid: both key widths (the grid decides), is_dense 0 / 1 (non-dense clouds carry a few NaN rows)."""
    x, leaf = _dense_case(case)
    if not is_dense:
        x = x.copy()
        x[::501, 1] = np.nan
    min_points = 1 if case.startswith("D") else 2
    with CloudMerger(max_batch_points=len(x)) as cm:
        cm.set_voxel(leaf, min_points, True)
        buf = cm.upload(x)
        cm.dev_voxelgrid(buf.ptr, len(x), is_dense=bool(is_dense))
        out = cm.fetch_batch_outputs()
    o = oracle.voxelgrid(x, [leaf] * 3, min_points, True, force64=True, is_dense=bool(is_dense))
    o.update(n_voxels=o["n"], n_survivors=len(x))
    st = out["stats"]
    cells = int(np.prod(o["div_b"].astype(np.int64)))
    want_bits = E.bits_for(cells) + (0 if is_dense else 1)     # non-finite points are keyed into a frame of their own
    assert st.device_error == 0 and st.frames == 1
    assert st.key_bits == want_bits and out["key_bytes"] == (4 if want_bits <= 32 else 8)
    assert st.sort_passes == max(1, -(-want_bits // 8))
    assert st.pcl_overflow == int(o["pcl_overflow"])
    check_voxels(out, out["frames"], [o], check_membership=bool(is_dense))
    assert_centroids_within_bound(out["voxel_xyzi"], o["centroid_f64"], x, o["point_idx"], o["idx"], o["count"], case)


def _box_frames(kind, F):
    """(frames [[(xyzi, dense)]], extrinsic, passes, leaf) of the K1 fused-key cases: a box that bounds x, y and z."""
    if kind.startswith("B"):
        with_int = kind == "B2"
        passes = [(a, BOX[a][0], BOX[a][1], 0) for a in range(3)] + ([(3, INT_WINDOW[0], INT_WINDOW[1], 0)] if with_int else [])
        frames = []
        for f in range(F):
            x = E.box_limit_cloud(400 + f, BOX_T, BOX, intensity_window=INT_WINDOW if with_int else None, n_random=20000)
            dense = f % 2
            if not dense:
                x[::113, 0] = np.nan
            frames.append([(x, dense)])
        return frames, E.identity_extrinsic(BOX_T), passes, 0.1 if with_int else 0.25
    if kind == "B-zero":
        passes = [(0, 0.0, 0.5, 0), (1, -1.0, 0.0, 0), (2, -1.0, 1.0, 0), (3, 0.0, 255.0, 0)]
        return ([[(E.signed_zero_subnormal_cloud(410 + f), 1)] for f in range(F)], E.identity_extrinsic((-0.0, -0.0, -0.0)),
                passes, 0.05)
    if kind.startswith("A"):
        leaf = float(kind[1:])
        k = 50 * leaf
        passes = [(0, -k, k, 0), (1, -k, k, 0), (2, -k, k, 0)]
        return [[(E.lattice_cloud(420 + f, leaf, n_lattice=40000, n_filler=20000), 1)] for f in range(F)], \
            E.identity_extrinsic((0, 0, 0)), passes, leaf
    if kind == "C":
        c = E.MAP_CENTRE
        passes = [(0, c[0] - 25.0, c[0] + 25.0, 0), (1, c[1] - 25.0, c[1] + 25.0, 0), (2, c[2] - 2.5, c[2] + 2.5, 0)]
        return [[(E.offset_cloud(430 + f, 0.05, n=80000), 1)] for f in range(F)], E.identity_extrinsic((0, 0, 0)), passes, 0.05
    raise ValueError(kind)


@pytest.mark.parametrize("kind", ["A0.1", "A0.035", "A0.333333", "A0.25", "B1", "B2", "B-zero", "C"])
def test_fused_box_keys_edges(gpu_ok, oracle, kind):
    """K1 keys the survivors on the crop box's grid (single-box predicate, BOX 1 without and BOX 2 with an intensity window)
    and the centroid pass re-bases them onto every frame's data grid: limits hit exactly and one ulp either side, -0.0
    against 0.0, subnormals, lattice points, kilometre offsets; three frames, dense and non-dense."""
    F = 3
    frames, m, passes, leaf = _box_frames(kind, F)
    total = sum(len(p) for fr in frames for p, _ in fr)
    with CloudMerger(max_sensors=1, max_batch_points=total, max_batch_frames=F) as cm:
        cm.set_extrinsic(0, m)
        cm.set_crop(passes)
        cm.set_voxel(leaf, 1, True)
        segs, per_frame = upload_segments(cm, frames, lambda f, s: PACKED)
        cm.run_batch(segs)
        out = cm.fetch_batch_outputs()
    o = [oracle.merge_frame(cds, passes, [leaf] * 3, 1, True, True) for cds in per_frame]
    st = out["stats"]
    assert st.device_error == 0 and st.frames == F and out["key_bytes"] == 4 and st.survivors > 0
    check_survivors(out, out["frames"], o)
    check_voxels(out, out["frames"], o)
    pts = [fo["survivor_xyzi"] for fo in o]
    _bound_check(out, out["frames"], o, pts)
    if kind.startswith("B"):   # the limits decide: some points on them survive, their one-ulp outside neighbours do not
        assert 0 < st.survivors < st.points_in


@pytest.mark.parametrize("F", [2, 3])
def test_box_grid_at_32_bits_with_frame_bits(gpu_ok, oracle, F):
    """A crop box whose grid needs 31 index bits: with 2 frames (one frame bit) the key is exactly 32 bits and K1 keys the
    survivors on the box grid; with 3 frames it would need 33 and crop_box_grid falls back -- the batch then sorts
    frame-segmented on the box's 31-bit bound. Either way every frame matches the oracle."""
    div = (2048, 1024, 1023)
    box = [(a, 0.0, float(div[a]) - 0.5, 0) for a in range(3)]
    fr = [[(E.grid_cloud(440 + f, div, n_filler=30000), 1)] for f in range(F)]
    total = sum(len(p) for x in fr for p, _ in x)
    with CloudMerger(max_sensors=1, max_batch_points=total, max_batch_frames=F) as cm:
        cm.set_extrinsic(0, E.identity_extrinsic((0, 0, 0)))
        cm.set_crop(box)
        cm.set_voxel(1.0, 1, True)
        segs, per_frame = upload_segments(cm, fr, lambda f, s: PACKED)
        cm.run_batch(segs)
        out = cm.fetch_batch_outputs()
    o = [oracle.merge_frame(cds, box, [1.0] * 3, 1, True, True) for cds in per_frame]
    st = out["stats"]
    assert E.bits_for(int(np.prod(np.asarray(div, np.int64)))) == 31
    assert st.device_error == 0 and st.frames == F and st.key_bytes == 4 and st.sort_passes == 4
    if F == 2:
        assert st.key_bits == 32 and out["key_idx_bits"] == 31     # frame bit + box index: the fused keys
    else:
        assert st.key_bits == out["key_idx_bits"] == 31             # segmented: no frame bits sorted
    check_survivors(out, out["frames"], o)
    check_voxels(out, out["frames"], o)


@pytest.mark.parametrize("case,F", [("A:0.1", 3), ("A:0.035", 3), ("C:0.05", 3), ("D:2p31", 2), ("D:2p31", 5),
                                    ("D:2p32", 3), ("D:2p32+", 2), ("D:2p32+", 4)])
def test_segmented_batch_edges(gpu_ok, oracle, case, F):
    """A z-only crop leaves the grid unbounded, so a batch of F frames plans its sort on the device: a voxel index of up to
    32 bits sorts frame-segmented (32-bit records, no frame bits); one of 33 bits needs 64-bit keys with the frame bits."""
    frames = []
    for f in range(F):
        x, leaf = _dense_case(case)
        x = np.concatenate([np.roll(x, 997 * f, axis=0), x[:97 * f]])   # frames of different sizes and orders, same grid
        frames.append([(x, 1)])
    z_only = [(2, -1e6, 1e6, 0)]
    total = sum(len(p) for fr in frames for p, _ in fr)
    with CloudMerger(max_sensors=1, max_batch_points=total, max_batch_frames=F) as cm:
        cm.set_extrinsic(0, E.identity_extrinsic((0, 0, 0)))
        cm.set_crop(z_only)
        cm.set_voxel(leaf, 1, True)
        segs, per_frame = upload_segments(cm, frames, lambda f, s: PACKED)
        cm.run_batch(segs)
        out = cm.fetch_batch_outputs()
    o = [oracle.merge_frame(cds, z_only, [leaf] * 3, 1, True, True) for cds in per_frame]
    st = out["stats"]
    idx_bits = max(E.bits_for(int(np.prod(fo["div_b"].astype(np.int64)))) for fo in o)
    assert st.device_error == 0 and st.frames == F and out["key_idx_bits"] == idx_bits
    if idx_bits <= 32:
        assert st.key_bytes == 4 and st.key_bits == idx_bits
    else:
        assert st.key_bytes == 8 and st.key_bits == idx_bits + E.bits_for(F)
    assert st.sort_passes == max(1, -(-st.key_bits // 8))
    check_survivors(out, out["frames"], o)
    check_voxels(out, out["frames"], o)
    _bound_check(out, out["frames"], o, [fo["survivor_xyzi"] for fo in o])


def _host_frames(kind, n_frames):
    """(clouds per frame, extrinsic, passes, leaf) of the host-path cases."""
    if kind == "B-box":
        passes = [(a, BOX[a][0], BOX[a][1], 0) for a in range(3)] + [(3, INT_WINDOW[0], INT_WINDOW[1], 0)]
        return [E.box_limit_cloud(500 + f, BOX_T, BOX, intensity_window=INT_WINDOW, n_random=8000) for f in range(n_frames)], \
            E.identity_extrinsic(BOX_T), passes, 0.1
    if kind == "B-rotated":
        m = E.rotated_extrinsic(0.7, (3.0, -2.0, 1.5), pitch=0.05)
        clouds = [E.lattice_cloud(510 + f, 0.1, n_lattice=10000, n_filler=10000) for f in range(n_frames)]
        lim = E.limits_from_data(np_oracle.transform(clouds[0], m.reshape(-1)))
        return clouds, m, [(a, lo, hi, 0) for a, lo, hi in lim], 0.1
    if kind == "A-zonly":
        return [E.lattice_cloud(520 + f, 0.035, n_lattice=12000, n_filler=8000) for f in range(n_frames)], \
            E.identity_extrinsic((0, 0, 0)), [(2, -1.0, 1.5, 0)], 0.035
    if kind == "C-km-extrinsic":
        m = E.rotated_extrinsic(-1.1, (2500.0, -3800.0, 35.0))
        return [E.lattice_cloud(530 + f, 0.05, n_lattice=12000, n_filler=12000) for f in range(n_frames)], m, \
            [(2, 33.0, 37.0, 0)], 0.05
    if kind == "D-guard":
        return [E.grid_cloud(540 + f, E.DIV_GUARD_ABOVE, n_filler=8000, inset=0.9) for f in range(n_frames)], \
            E.identity_extrinsic((0, 0, 0)), [(2, -1.0, 2000.0, 0)], 1.0
    raise ValueError(kind)


@pytest.mark.parametrize("kind", ["B-box", "B-rotated", "A-zonly", "C-km-extrinsic", "D-guard"])
@pytest.mark.parametrize("pcl_like", [False, True])
def test_host_path_plain_captured_replayed(gpu_ok, oracle, kind, pcl_like):
    """cm_merge_frame three times per configuration: the plain enqueue, the CUDA-graph capture and its replay, each on new
    points, each against the oracle (in overflow mode 1 a frame PCL refuses comes back as its cropped cloud)."""
    clouds, m, passes, leaf = _host_frames(kind, 3)
    n = max(len(c) for c in clouds)
    with CloudMerger(max_sensors=1, max_points_per_sensor=n, frames_in_flight=1) as cm:
        cm.set_extrinsic(0, m)
        cm.set_crop(passes)
        cm.set_voxel(leaf, 1, True)
        cm.set_overflow_mode(pcl_like)
        for f, x in enumerate(clouds):
            cm.submit_cloud(0, x, len(x), make_layout())
            r = cm.merge_frame(capacity=n)
            o = oracle.merge_frame([cloud_dict(x, m)], passes, [leaf] * 3, 1, True, not pcl_like)
            assert (r.survivor_src == o["survivor_src"]).all(), (kind, f)
            assert_bit_equal(r.survivor_xyzi, o["survivor_xyzi"], "%s frame %d survivors" % (kind, f))
            assert bool(r.info.pcl_overflow) == o["pcl_overflow"]
            if o["returned_input"]:
                assert_bit_equal(r.voxel_xyzi, o["survivor_xyzi"], "refused frame = its cropped cloud")
                continue
            assert list(r.info.div_b) == o["div_b"].tolist() and list(r.info.min_b) == o["min_b"].tolist()
            assert (r.voxel_idx.astype(np.int64) == o["idx"]).all() and (r.voxel_count == o["count"]).all(), (kind, f)
            assert_bit_equal(r.voxel_xyzi, o["centroid"], "%s frame %d centroids" % (kind, f))
            assert_centroids_within_bound(r.voxel_xyzi, o["centroid_f64"], o["survivor_xyzi"], o["point_idx"], o["idx"],
                                          o["count"], kind)


@pytest.mark.parametrize("case", ["A:0.05", "C:0.05"])
def test_global_bounds_edges(gpu_ok, case):
    """cm_set_voxel_bounds: the grid comes from a box wider than the data (a block of a partitioned cloud), checked against
    the numpy restatement with the same bounds."""
    x, leaf = _dense_case(case)
    c = np.asarray(E.MAP_CENTRE if case.startswith("C") else (0.0, 0.0, 0.0))
    mn, mx = (c - 80.0).astype(np.float32), (c + 70.0).astype(np.float32)
    with CloudMerger(max_batch_points=len(x)) as cm:
        cm.set_voxel(leaf, 1, True)
        cm.set_voxel_bounds(mn, mx)
        buf = cm.upload(x)
        cm.dev_voxelgrid(buf.ptr, len(x))
        out = cm.fetch_batch_outputs()
    o = np_oracle.voxelgrid(x, [leaf] * 3, 1, True, True, bounds=(mn, mx))
    fi = out["frames"][0]
    assert out["stats"].device_error == 0
    assert list(fi.min_b) == o["min_b"].tolist() and list(fi.div_b) == o["div_b"].tolist()
    assert (out["voxel_idx"].astype(np.int64) == o["idx"]).all() and (out["voxel_count"] == o["count"]).all()
    assert_centroids_within_bound(out["voxel_xyzi"], o["centroid_f64"], x, o["point_idx"], o["idx"], o["count"], case)


# ---- the key range: documented errors, and overflow mode 1 -----------------------------------------------------------------
def _far_return_cloud(seed, distance):
    """A sensor cloud of a few metres plus one bogus return `distance` metres away on x."""
    x = E.lattice_cloud(seed, 0.05, n_lattice=4000, n_filler=4000, k_span=40)
    x[17, :3] = (distance, 0.5, 0.25)
    return x


def test_key_range_errors_and_recovery(gpu_ok, oracle):
    """Overflow mode 0: a frame with more than 2^21 cells on an axis, or a cell origin at 2^30, raises CM_E_KEY_RANGE -- it
    never returns wrong voxels -- and the handle then gives oracle-exact results on the next frames, a replayed graph
    included. (2^21 cells on an axis and the largest float32 origin below 2^30 are accepted: test_dense_voxelgrid_edges.)"""
    z_only = [(2, -1e12, 1e12, 0)]
    good = [E.lattice_cloud(600 + f, 0.1, n_lattice=5000, n_filler=5000) for f in range(3)]
    bad = [E.grid_cloud(610, ((1 << 21) + 1, 3, 2), n_filler=3000),                       # 2^21 + 1 cells on x, no guard trip
           E.grid_cloud(611, (4, 5, 6), n_filler=3000, origin=(E.ORIGIN_BEYOND, 0.0, 0.0)),
           E.grid_cloud(612, (4, 5, 6), n_filler=3000, origin=(-E.ORIGIN_BEYOND - 64.0, 0.0, 0.0))]
    n = max(len(c) for c in good + bad)
    with CloudMerger(max_sensors=1, max_points_per_sensor=n, frames_in_flight=1, max_batch_points=n) as cm:
        cm.set_extrinsic(0, E.identity_extrinsic((0, 0, 0)))
        cm.set_crop(z_only)
        cm.set_voxel(1.0, 1, True)
        for x in bad:
            cm.submit_cloud(0, x, len(x), make_layout())
            with pytest.raises(CloudMergerError) as e:
                cm.merge_frame(capacity=n)
            assert e.value.code == _lib.CM_E_KEY_RANGE
            buf = cm.upload(x)
            with pytest.raises(CloudMergerError) as e:
                cm.dev_voxelgrid(buf.ptr, len(x))
                cm.fetch_batch_outputs()
            assert e.value.code == _lib.CM_E_KEY_RANGE
            buf.free()
        cm.set_voxel(0.1, 1, True)
        for f, x in enumerate(good):   # plain, captured, replayed
            cm.submit_cloud(0, x, len(x), make_layout())
            r = cm.merge_frame(capacity=n)
            o = oracle.merge_frame([cloud_dict(x, E.identity_extrinsic((0, 0, 0)))], z_only, [0.1] * 3, 1, True, True)
            assert (r.survivor_src == o["survivor_src"]).all()
            assert (r.voxel_idx.astype(np.int64) == o["idx"]).all() and (r.voxel_count == o["count"]).all(), f
            assert_bit_equal(r.voxel_xyzi, o["centroid"], "frame %d after the errors" % f)


def test_overflow_mode_1_returns_the_cropped_cloud_beyond_the_key_range(gpu_ok, oracle):
    """Config 1's z-only crop at leaf 0.01 with one bogus return 30 km away: more than 2^21 cells on x, and PCL's guard trips,
    so PCL returns the cropped cloud. Overflow mode 1 must do the same (no CM_E_KEY_RANGE); mode 0 reports the key range.
    The mode toggles between frames of one shape, across graph capture and replay."""
    z_only = [(2, -1.0, 2.0, 0)]
    leaf = 0.01
    clouds = [_far_return_cloud(700 + f, 30000.0) for f in range(7)]
    n = len(clouds[0])
    with CloudMerger(max_sensors=1, max_points_per_sensor=n, frames_in_flight=1) as cm:
        cm.set_extrinsic(0, E.identity_extrinsic((0, 0, 0)))
        cm.set_crop(z_only)
        cm.set_voxel(leaf, 1, True)
        # 1 1 1: plain, capture, replay; 0: must not replay the mode-1 graph; 1 1 1 again
        for f, (x, mode) in enumerate(zip(clouds, (1, 1, 1, 0, 1, 1, 1))):
            cm.set_overflow_mode(bool(mode))
            cm.submit_cloud(0, x, len(x), make_layout())
            o = oracle.merge_frame([cloud_dict(x, E.identity_extrinsic((0, 0, 0)))], z_only, [leaf] * 3, 1, True, False)
            grid = np_oracle.voxelgrid(o["survivor_xyzi"], [leaf] * 3, 1, True, False)
            assert o["returned_input"] and grid["pcl_overflow"] and grid["div_b"][0] > (1 << 21)
            if mode == 0:
                with pytest.raises(CloudMergerError) as e:
                    cm.merge_frame(capacity=n)
                assert e.value.code == _lib.CM_E_KEY_RANGE
                continue
            r = cm.merge_frame(capacity=n)
            assert r.info.pcl_overflow
            assert (r.survivor_src == o["survivor_src"]).all()
            assert_bit_equal(r.voxel_xyzi, o["survivor_xyzi"], "frame %d: PCL's output is the cropped cloud" % f)
            assert (r.voxel_count == 1).all()
