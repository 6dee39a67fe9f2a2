"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the CPU oracle on the same seeded inputs.

Bar (north_star): bit-exact surviving-point indices and coordinates, voxel membership, counts and output order;
centroids within 1e-5 relative of the double-precision oracle (and, because the radix sort is stable, bit-equal to the
oracle's float accumulation in ascending point order).
"""
import numpy as np
import pytest

from cloud_merger_b200 import CloudMerger, CloudMergerError, _lib, make_layout, synth

from helpers import (assert_bit_equal, assert_centroids_close, check_survivors, check_voxels, cloud_dict, known_answer,
                     upload_segments)

pytestmark = pytest.mark.gpu

LAYOUTS = {
    "packed16": (16, 0, 4, 8, 12),
    "pcl32": (32, 0, 4, 8, 16),
    "aligned48": (48, 8, 12, 16, 36),
    "noint20": (20, 4, 8, 12, -1),
    "velodyne22": (22, 0, 4, 8, 12),
    "livox18": (18, 0, 4, 8, 12),
    "odd19": (19, 3, 7, 11, 15),
    "bytes100": (101, 1, 5, 9, 13),
}


def _layout(t, dense=1):
    return make_layout(t[0], t[1], t[2], t[3], t[4], dense)


def _oracle_frames(oracle, per_frame, passes, leaf, min_points, downsample_all=True):
    return [oracle.merge_frame(cds, passes, leaf, min_points, downsample_all, True) for cds in per_frame]


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("min_points", [1, 2])
def test_known_answer_host_path(gpu_ok, min_points):
    """The hand-computed vector of tests/golden/known_answer.json through submit_cloud / merge_frame."""
    ka = known_answer()
    e = ka["expected"]
    with CloudMerger(max_sensors=2, max_points_per_sensor=16) as cm:
        cm.set_extrinsic(0, np.array(ka["extrinsics_row_major_3x4"]["A"], np.float32))
        cm.set_extrinsic(1, np.array(ka["extrinsics_row_major_3x4"]["B"], np.float32))
        cm.set_crop([tuple(p) for p in ka["crop_passes"]])
        cm.set_voxel(ka["leaf"], min_points, True)
        cm.submit_cloud(0, ka["A"], 4, make_layout(is_dense=1), stamp=5)
        cm.submit_cloud(1, ka["B"], 4, make_layout(is_dense=0), stamp=9)
        r = cm.merge_frame(capacity=8)
    assert r.survivor_src.tolist() == e["survivor_src"]
    assert_bit_equal(r.survivor_xyzi[:, :3], np.array(e["survivor_xyz"], np.float32), "survivors")
    assert list(r.info.min_b) == e["min_b"] and list(r.info.max_b) == e["max_b"] and list(r.info.div_b) == e["div_b"]
    ex = e["min_points_%d" % min_points]
    assert r.voxel_idx.tolist() == ex["idx"] and r.voxel_count.tolist() == ex["count"]
    assert_bit_equal(r.voxel_xyzi, np.array(ex["centroid"], np.float32), "centroids")
    assert r.used_mask == 3 and r.stamp == 9 and not r.info.pcl_overflow


@pytest.mark.parametrize("name", list(LAYOUTS))
@pytest.mark.parametrize("dense", [1, 0])
def test_transform_crop_layouts(gpu_ok, oracle, name, dense):
    """K1 alone on every record layout (16-byte fast path, PCL 32-byte, 4-byte aligned, TMA-staged unaligned, byte
    fallback), ragged sizes around the 2048-point tile, with and without non-finite points."""
    lt = LAYOUTS[name]
    sizes = [0, 1, 31, 2047, 2048, 2049, 5000, 12345]
    rng = np.random.default_rng(42)
    sensors = []
    for s, n in enumerate(sizes):
        p = synth.lidar_cloud(77, s, 0, 1, max(n, 1))[:n]
        if not dense and n:
            bad = rng.random(n) < 0.02
            p[bad, rng.integers(0, 3)] = np.nan
            if n > 10:
                p[3, 1] = np.inf
        sensors.append((p, dense))
    with CloudMerger(max_sensors=len(sizes), max_batch_points=sum(sizes), max_batch_frames=1) as cm:
        for s in range(len(sizes)):
            cm.set_extrinsic(s, synth.extrinsic(s, len(sizes)))
        cm.set_crop(synth.ROI_BOX)
        segs, per_frame = upload_segments(cm, [sensors], lambda f, s: lt)
        cm.dev_transform_crop(segs)
        out = cm.fetch_batch_outputs()
        o = _oracle_frames(oracle, per_frame, synth.ROI_BOX, [0.1] * 3, 1)
        check_survivors(out, out["frames"], o)
        assert out["stats"].survivors == o[0]["n_survivors"] > 100
        assert out["stats"].points_in == sum(sizes)


def test_transform_crop_mixed_layouts_and_pass_kinds(gpu_ok, oracle):
    """Sensors with different layouts in one frame; negative pass and an intensity pass; limits sitting exactly on data."""
    names = ["packed16", "velodyne22", "pcl32", "livox18", "odd19", "aligned48"]
    sensors = [(synth.lidar_cloud(5, s, 1, 16, 512, nan_frac=0.01), 0) for s in range(len(names))]
    some = np.sort(sensors[0][0][:, 2])
    passes = [(2, float(some[100]), float(some[-100]), 0), (0, -2.0, 2.0, 1), (3, 10.0, 200.0, 0), (1, -40.0, 40.0, 0)]
    with CloudMerger(max_sensors=len(names), max_batch_points=len(names) * 8192) as cm:
        for s in range(len(names)):
            cm.set_extrinsic(s, synth.extrinsic(s, len(names)))
        cm.set_crop(passes)
        segs, per_frame = upload_segments(cm, [sensors], lambda f, s: LAYOUTS[names[s]])
        cm.dev_transform_crop(segs)
        out = cm.fetch_batch_outputs()
        o = _oracle_frames(oracle, per_frame, passes, [0.1] * 3, 1)
        check_survivors(out, out["frames"], o)
        assert 0 < out["stats"].survivors < out["stats"].points_in


def test_no_crop_keeps_everything_and_voxel_skips_invalid(gpu_ok, oracle):
    """Zero passes = plain cloud_fusion concat (CloudFusionNode.h:59-72): every point survives, non-finite ones included
    (left untransformed for a non-dense cloud); VoxelGrid then skips them like PCL does for !is_dense."""
    sensors = [(synth.lidar_cloud(6, s, 0, 8, 700, nan_frac=0.03), 0) for s in range(3)]
    with CloudMerger(max_sensors=3, max_batch_points=3 * 5600) as cm:
        for s in range(3):
            cm.set_extrinsic(s, synth.extrinsic(s, 3))
        cm.set_crop([])
        cm.set_voxel(0.5, 1, True)
        segs, per_frame = upload_segments(cm, [sensors], lambda f, s: LAYOUTS["packed16"])
        cm.run_batch(segs)
        out = cm.fetch_batch_outputs()
        o = _oracle_frames(oracle, per_frame, [], [0.5] * 3, 1)
        assert out["stats"].survivors == 3 * 5600
        check_survivors(out, out["frames"], o)
        assert np.isnan(out["survivor_xyzi"]).any()
        check_voxels(out, out["frames"], o, check_membership=False)
        # membership: invalid points carry the sentinel frame and are sorted to the end
        n_bad = int((~np.isfinite(out["survivor_xyzi"][:, :3]).all(axis=1)).sum())
        tail = out["sorted_point"][len(out["sorted_point"]) - n_bad:]
        assert (~np.isfinite(out["survivor_xyzi"][tail, :3]).all(axis=1)).all()


@pytest.mark.parametrize("leaf,min_points", [(1.0, 1), (0.5, 2), (0.2, 3), (0.1, 2), (0.05, 1), (0.02, 1), (0.01, 2)])
def test_voxelgrid_only_leaf_sweep(gpu_ok, oracle, leaf, min_points):
    """VoxelGrid alone (cm_dev_voxelgrid) across occupancy regimes; the fine leaves exceed PCL's INT32 cell limit and run
    on 64-bit keys (oracle force64)."""
    x = synth.uniform_cloud(21, 300000, extent=(200.0, 200.0, 10.0))
    x[:50000] = synth.uniform_cloud(22, 50000, extent=(6.0, 6.0, 2.0))  # a dense clump: long runs
    with CloudMerger(max_batch_points=len(x)) as cm:
        cm.set_voxel(leaf, min_points, True)
        buf = cm.upload(x)
        cm.dev_voxelgrid(buf.ptr, len(x))
        out = cm.fetch_batch_outputs()
    o = oracle.voxelgrid(x, [leaf] * 3, min_points, True, force64=True)
    o.update(n_voxels=o["n"], n_survivors=len(x))
    assert out["stats"].pcl_overflow == int(o["pcl_overflow"])
    assert out["key_bytes"] == (4 if out["stats"].key_bits <= 32 else 8)
    worst = check_voxels(out, out["frames"], [o])
    assert worst <= 1e-5


def test_voxelgrid_degenerate_inputs(gpu_ok, oracle):
    with CloudMerger(max_batch_points=4096) as cm:
        cm.set_voxel(0.1, 1, True)
        # a single point, all points identical, all points invalid, empty
        for x in (np.array([[1, 2, 3, 4]], np.float32), np.tile(np.array([[0.5, -0.5, 0.25, 9]], np.float32), (3000, 1)),
                  np.full((100, 4), np.nan, np.float32), np.zeros((0, 4), np.float32)):
            buf = cm.upload(x if len(x) else np.zeros((1, 4), np.float32))
            cm.dev_voxelgrid(buf.ptr, len(x), is_dense=False)
            out = cm.fetch_batch_outputs()
            o = oracle.voxelgrid(x, [0.1] * 3, 1, True, force64=True, is_dense=False)
            assert out["stats"].voxels_out == o["n"]
            if o["n"]:
                assert (out["voxel_count"] == o["count"]).all()
                assert_bit_equal(out["voxel_xyzi"], o["centroid"], "centroid")


def test_downsample_all_false_and_pcl_record_layout(gpu_ok, oracle):
    x = synth.uniform_cloud(3, 20000, extent=(10.0, 10.0, 2.0))
    with CloudMerger(max_batch_points=len(x), out_point_step=32) as cm:
        cm.set_voxel(0.25, 2, False)
        buf = cm.upload(x)
        cm.dev_voxelgrid(buf.ptr, len(x))
        out = cm.fetch_batch_outputs()
    o = oracle.voxelgrid(x, [0.25] * 3, 2, False, force64=True)
    rec = out["voxel_records"]
    assert rec.shape[1] == 8 and (rec[:, 3] == 1.0).all() and (rec[:, 5:] == 0).all() and (rec[:, 4] == 0).all()
    assert_bit_equal(out["voxel_xyzi"], o["centroid"], "centroid (xyz only)")


def test_batch_of_frames_matches_per_frame_oracle(gpu_ok, oracle):
    """F frames x S sensors in one device-resident batch: frame-major keys, per-frame grids, per-frame slices."""
    F, S = 5, 3
    frames = [[(synth.lidar_cloud(31, s, f, 16, 300 + 37 * f + 11 * s), 1) for s in range(S)] for f in range(F)]
    frames[2][1] = (np.zeros((0, 4), np.float32), 1)          # an empty cloud inside a frame
    frames[3] = [(np.full((10, 4), 1e6, np.float32), 1)] * S  # a frame whose points are all cropped away
    total = sum(len(p) for fr in frames for p, _ in fr)
    with CloudMerger(max_sensors=S, max_batch_points=total, max_batch_frames=F) as cm:
        for s in range(S):
            cm.set_extrinsic(s, synth.extrinsic(s, S))
        cm.set_crop(synth.ROI_BOX)
        cm.set_voxel(0.1, 2, True)
        segs, per_frame = upload_segments(cm, frames, lambda f, s: LAYOUTS["packed16" if (f + s) % 2 else "pcl32"])
        cm.run_batch(segs)
        out = cm.fetch_batch_outputs()
        o = _oracle_frames(oracle, per_frame, synth.ROI_BOX, [0.1] * 3, 2)
        assert out["stats"].frames == F and out["key_bytes"] == 4
        check_survivors(out, out["frames"], o)
        check_voxels(out, out["frames"], o)
        assert out["frames"][3].survivor_begin == out["frames"][3].survivor_end
        assert cm.launch_count() >= 5


@pytest.mark.parametrize("cfg,nan_frac", [("cfg1", 0.0), ("cfg2", 0.0), ("cfg2", 0.005)])
def test_config_shapes_host_path(gpu_ok, oracle, cfg, nan_frac):
    """BASELINE configs 1 and 2 at full size through the host path (submit per sensor, merge), mixed record layouts."""
    c = synth.CONFIGS[cfg]
    clouds, mats = synth.frame_clouds(cfg, 1000 * int(cfg[-1]), 0, nan_frac)
    S, n = c["sensors"], len(clouds[0])
    lts = [LAYOUTS["packed16"], LAYOUTS["pcl32"], LAYOUTS["velodyne22"], LAYOUTS["livox18"]]
    dense = 0 if nan_frac else 1
    with CloudMerger(max_sensors=S, max_points_per_sensor=n, max_point_step=32) as cm:
        cds = []
        for s in range(S):
            cm.set_extrinsic(s, mats[s])
            lt = lts[s % len(lts)]
            data = synth.pack_cloud(clouds[s], *lt)
            cm.submit_cloud(s, data, n, _layout(lt, dense), stamp=100 + s)
            cds.append(cloud_dict(clouds[s], mats[s][:3], dense, *lt))
        cm.set_crop(c["passes"])
        cm.set_voxel(c["leaf"], c["min_points"], True)
        r = cm.merge_frame(capacity=S * n)
        st = cm.stats()
    o = oracle.merge_frame(cds, c["passes"], [c["leaf"]] * 3, c["min_points"], True, True)
    assert len(r.survivor_src) == o["n_survivors"] and (r.survivor_src == o["survivor_src"]).all()
    assert_bit_equal(r.survivor_xyzi, o["survivor_xyzi"], "survivors")
    assert len(r.voxel_idx) == o["n_voxels"] > 1000
    assert (r.voxel_idx.astype(np.int64) == o["idx"]).all() and (r.voxel_count == o["count"]).all()
    assert_bit_equal(r.voxel_xyzi, o["centroid"], "centroid vs float oracle")
    assert_centroids_close(r.voxel_xyzi, o["centroid_f64"], "centroid vs f64 oracle")
    assert r.stamp == 100 + S - 1 and r.used_mask == (1 << S) - 1
    assert st.survivors == o["n_survivors"] and st.voxels_out == o["n_voxels"]


def test_pipelined_frames_and_optional_sensor(gpu_ok, oracle):
    """Three frames in flight (merge_frame_async / wait_frame); a sensor missing from one frame is skipped like the
    reference's optional top sensor (pc_preprocessing_main.cpp:134-136)."""
    S, n = 3, 4000
    with CloudMerger(max_sensors=S, max_points_per_sensor=n, frames_in_flight=3) as cm:
        mats = [synth.extrinsic(s, S) for s in range(S)]
        for s in range(S):
            cm.set_extrinsic(s, mats[s])
        cm.set_crop(synth.ROI_BOX)
        cm.set_voxel(0.2, 1, True)
        tickets, expect = [], []
        for f in range(3):
            cds = []
            for s in range(S):
                if f == 1 and s == 2:
                    continue
                p = synth.lidar_cloud(55, s, f, 8, n // 8)
                cm.submit_cloud(s, p, len(p), make_layout(), stamp=f)
                cds.append(cloud_dict(p, mats[s][:3]))
            tickets.append(cm.merge_frame_async())
            expect.append(oracle.merge_frame(cds, synth.ROI_BOX, [0.2] * 3, 1, True, True))
        with pytest.raises(CloudMergerError) as e:   # every slot is now in flight
            cm.submit_cloud(0, np.zeros((1, 4), np.float32), 1, make_layout())
        assert e.value.code == _lib.CM_E_CAPACITY
        for f in (0, 1, 2):
            r = cm.wait_frame(tickets[f], capacity=S * n)
            o = expect[f]
            assert r.used_mask == (0b011 if f == 1 else 0b111)
            assert (r.survivor_src == o["survivor_src"]).all()
            assert (r.voxel_idx.astype(np.int64) == o["idx"]).all() and (r.voxel_count == o["count"]).all()
            assert_bit_equal(r.voxel_xyzi, o["centroid"], "frame %d" % f)


def test_concurrent_sensor_callbacks_and_frame_graphs(gpu_ok, oracle):
    """The reference runs its six sensor callbacks on ros::AsyncSpinner(6) and fuses on the main thread
    (pc_preprocessing_main.cpp:513, :574-578): cm_submit_cloud from one thread per sensor, concurrently, then the merge.
    Twelve frames of the same shape also take the host path through its plain / captured / replayed-graph stages; every
    frame must match the oracle."""
    import threading
    S, rings, az = 6, 16, 128
    n = rings * az
    passes, leaf, mp = synth.ROI_BOX, 0.1, 2
    with CloudMerger(max_sensors=S, max_points_per_sensor=n, frames_in_flight=2) as cm:
        mats = [synth.extrinsic(s, S) for s in range(S)]
        for s in range(S):
            cm.set_extrinsic(s, mats[s])
        cm.set_crop(passes)
        cm.set_voxel(leaf, mp, True)
        for f in range(12):
            clouds = [synth.lidar_cloud(77, s, f, rings, az) for s in range(S)]
            errs = []

            def callback(s):
                try:
                    cm.submit_cloud(s, clouds[s], n, make_layout(), stamp=100 + f)
                except Exception as e:  # noqa: BLE001
                    errs.append(e)
            th = [threading.Thread(target=callback, args=(s,)) for s in range(S)]
            for t in th:
                t.start()
            for t in th:
                t.join()
            assert not errs, errs
            r = cm.merge_frame(capacity=S * n)
            o = oracle.merge_frame([cloud_dict(c, m[:3]) for c, m in zip(clouds, mats)], passes, [leaf] * 3, mp, True, True)
            assert r.used_mask == (1 << S) - 1 and r.stamp == 100 + f
            assert (r.survivor_src == o["survivor_src"]).all(), "frame %d" % f
            assert_bit_equal(r.survivor_xyzi, o["survivor_xyzi"], "frame %d survivors" % f)
            assert (r.voxel_idx.astype(np.int64) == o["idx"]).all() and (r.voxel_count == o["count"]).all(), "frame %d" % f
            assert_bit_equal(r.voxel_xyzi, o["centroid"], "frame %d centroids" % f)


def test_submit_clouds_pinned_matches_single_submits(gpu_ok, oracle):
    """cm_submit_clouds_pinned == one cm_submit_cloud_pinned per cloud, whether or not the clouds are adjacent in host
    memory (adjacent clouds of consecutive sensors travel as one copy), with ragged sizes and a skipped sensor id."""
    from cloud_merger_b200 import host_alloc
    S, cap = 4, 16 * 512
    sizes = [cap, cap - 37 * 16 // 16, 1234, cap]
    passes, leaf, mp = [(2, -0.5, 3.0, 0), (0, -15.0, 60.0, 0)], 0.1, 2
    arena, addr = host_alloc(S * cap * 16 + 4096)
    clouds, addrs, off = [], [], 0
    for s in range(S):
        c = synth.lidar_cloud(555, s, 0, 16, 512)[:sizes[s]]
        if s == 3:
            off += 256  # a gap: the last cloud is not adjacent to its predecessor
        arena[off:off + c.nbytes] = c.view(np.uint8).reshape(-1)
        clouds.append(c); addrs.append(addr + off)
        off += c.nbytes
    with CloudMerger(max_sensors=6, max_points_per_sensor=cap, frames_in_flight=2) as cm:
        ids = [0, 1, 2, 4]  # sensor 3 is never submitted: 0-1-2 form one run, 4 stands alone (and is not adjacent anyway)
        for s, sid in enumerate(ids):
            cm.set_extrinsic(sid, synth.extrinsic(s, S))
        cm.set_crop(passes); cm.set_voxel(leaf, mp, True)
        cm.submit_clouds_pinned(ids, addrs, sizes, [make_layout()] * S, stamps=[7, 8, 9, 10])
        got = cm.merge_frame(capacity=S * cap)
        for s, sid in enumerate(ids):
            cm.submit_cloud(sid, clouds[s], sizes[s], make_layout(), stamp=7 + s)
        ref = cm.merge_frame(capacity=S * cap)
        mats = [cm.get_extrinsic(sid) for sid in ids]
    assert got.stamp == ref.stamp == 10
    assert (got.survivor_src == ref.survivor_src).all() and len(got.survivor_src) > 1000
    assert_bit_equal(got.survivor_xyzi, ref.survivor_xyzi, "survivors")
    assert (got.voxel_idx == ref.voxel_idx).all() and (got.voxel_count == ref.voxel_count).all()
    assert_bit_equal(got.voxel_xyzi, ref.voxel_xyzi, "centroids")
    o = oracle.merge_frame([cloud_dict(c, m) for c, m in zip(clouds, mats)], passes, [leaf] * 3, mp, True, True)
    assert (got.survivor_src == o["survivor_src"]).all()
    assert (got.voxel_idx.astype(np.int64) == o["idx"]).all()


def test_pcl_overflow_modes(gpu_ok, oracle):
    """Leaf too small for the extent: PCL 1.8.1 returns the input unchanged (mode 1); the default carries on in 64 bits."""
    p = synth.uniform_cloud(8, 5000, extent=(300.0, 300.0, 20.0))
    for pcl_like in (False, True):
        with CloudMerger(max_sensors=1, max_points_per_sensor=len(p)) as cm:
            cm.set_crop([])
            cm.set_voxel(0.01, 1, True)
            cm.set_overflow_mode(pcl_like)
            cm.submit_cloud(0, p, len(p), make_layout())
            r = cm.merge_frame(capacity=len(p))
        assert r.info.pcl_overflow
        if pcl_like:
            o = oracle.voxelgrid(p, [0.01] * 3, 1, True, force64=False)
            assert o["returned_input"] and len(r.voxel_xyzi) == len(p)
            assert_bit_equal(r.voxel_xyzi, p, "output = input")
        else:
            o = oracle.voxelgrid(p, [0.01] * 3, 1, True, force64=True)
            assert (r.voxel_idx.astype(np.int64) == o["idx"]).all()
            assert_bit_equal(r.voxel_xyzi, o["centroid"], "64-bit path")


def test_error_behaviour(gpu_ok):
    with CloudMerger(max_sensors=2, max_points_per_sensor=100, max_point_step=16) as cm:
        with pytest.raises(CloudMergerError) as e:
            cm.submit_cloud(0, np.zeros((101, 4), np.float32), 101, make_layout())
        assert e.value.code == _lib.CM_E_CAPACITY
        with pytest.raises(CloudMergerError) as e:
            cm.submit_cloud(0, np.zeros((10, 8), np.float32), 10, make_layout(32, 0, 4, 8, 16))
        assert e.value.code == _lib.CM_E_CAPACITY
        with pytest.raises(CloudMergerError) as e:
            cm.submit_cloud(0, np.zeros((10, 4), np.float32), 10, make_layout(16, 0, 4, 14, 12))
        assert e.value.code == _lib.CM_E_INVALID
        with pytest.raises(CloudMergerError) as e:
            cm.submit_cloud(5, np.zeros((10, 4), np.float32), 10, make_layout())
        assert e.value.code == _lib.CM_E_INVALID
        with pytest.raises(CloudMergerError) as e:
            cm.merge_frame(capacity=10)
        assert e.value.code == _lib.CM_E_NOT_READY
        cm.set_crop([])
        cm.set_voxel(0.1, 1, True)
        cm.submit_cloud(0, np.arange(40, dtype=np.float32).reshape(10, 4), 10, make_layout())
        with pytest.raises(CloudMergerError) as e:   # caller buffer too small: reports instead of overrunning
            cm.merge_frame(capacity=3)
        assert e.value.code == _lib.CM_E_CAPACITY


def test_full_size_batch_properties(gpu_ok, oracle):
    """cfg 2 at bench size (16 frames x 4 x 128k points) checked through size-independent properties, plus an exact
    comparison of two of its frames with the oracle."""
    c = synth.CONFIGS["cfg2"]
    F, S = 16, c["sensors"]
    n = c["rings"] * c["azimuth"]
    with CloudMerger(max_sensors=S, max_batch_points=F * S * n, max_batch_frames=F) as cm:
        mats = [synth.extrinsic(s, S) for s in range(S)]
        for s in range(S):
            cm.set_extrinsic(s, mats[s])
        cm.set_crop(c["passes"])
        cm.set_voxel(c["leaf"], c["min_points"], True)
        frames = [[(synth.lidar_cloud(2000, s, f, c["rings"], c["azimuth"]), 1) for s in range(S)] for f in range(F)]
        segs, per_frame = upload_segments(cm, frames, lambda f, s: LAYOUTS["packed16"])
        cm.run_batch(segs)
        out = cm.fetch_batch_outputs()
        st = out["stats"]
        assert st.points_in == F * S * n and st.frames == F and st.device_error == 0
        keys = out["sorted_key"]
        assert (keys[1:] >= keys[:-1]).all(), "keys must be globally sorted (frame-major)"
        assert np.array_equal(np.sort(out["sorted_point"]), np.arange(st.survivors, dtype=np.uint32)), "a permutation"
        # every voxel's count is the length of its run of equal keys; dropped runs are the short ones
        uniq, cnt = np.unique(keys, return_counts=True)
        kept = cnt >= c["min_points"]
        assert kept.sum() == st.voxels_out and (out["voxel_count"] == cnt[kept]).all()
        # centroids lie inside their voxel (up to rounding at the faces)
        fi = out["frames"]
        for f in (0, F - 1):
            v0, v1 = fi[f].voxel_begin, fi[f].voxel_end
            idx = out["voxel_idx"][v0:v1].astype(np.int64)
            d0, d1 = fi[f].div_b[0], fi[f].div_b[1]
            ijk = np.stack([idx % d0, (idx // d0) % d1, idx // (d0 * d1)], axis=1) + np.array(fi[f].min_b)
            cell = np.floor(out["voxel_xyzi"][v0:v1, :3].astype(np.float64) / c["leaf"] + 1e-4)
            assert np.abs(cell - ijk).max() <= 1
        o = [oracle.merge_frame(per_frame[f], c["passes"], [c["leaf"]] * 3, c["min_points"], True, True) for f in (0, F - 1)]
        sel = [fi[0], fi[F - 1]]
        sub = dict(out)
        # compare frames 0 and F-1 exactly
        for k, (f, fo) in enumerate(zip((0, F - 1), o)):
            s0, s1, v0, v1 = sel[k].survivor_begin, sel[k].survivor_end, sel[k].voxel_begin, sel[k].voxel_end
            assert (out["survivor_src"][s0:s1] == fo["survivor_src"]).all()
            assert_bit_equal(out["survivor_xyzi"][s0:s1], fo["survivor_xyzi"], "frame %d survivors" % f)
            assert (out["voxel_idx"][v0:v1].astype(np.int64) == fo["idx"]).all()
            assert (out["voxel_count"][v0:v1] == fo["count"]).all()
            assert_bit_equal(out["voxel_xyzi"][v0:v1], fo["centroid"], "frame %d centroids" % f)
        del sub


# ---- round 2: every sort instantiation and every BASELINE config at size ------------------------------------------------
def _voxel_only(cm, x, leaf, min_points):
    cm.set_voxel(leaf, min_points, True)
    buf = cm.upload(x)
    cm.dev_voxelgrid(buf.ptr, len(x))
    out = cm.fetch_batch_outputs()
    buf.free()
    return out


@pytest.mark.parametrize("dense_points", [20, 5000, 700001])
def test_one_voxel_holding_most_of_the_cloud(gpu_ok, oracle, dense_points):
    """A voxel with far more points than a centroid tile (sensors that report invalid returns as zeros put them all into
    the voxel at the origin): its run spans hundreds of tiles and is finished by the whole CTA (finish_tail_run), in PCL's
    strictly sequential float order -- bit-equal to the float oracle -- and in milliseconds, not the second a lone thread
    took. (20 points: the hand-over threshold is not reached; 5000: a few tiles.)"""
    rng = np.random.default_rng(31)
    x = synth.uniform_cloud(91, 300000, extent=(60.0, 60.0, 6.0))
    blob = np.empty((dense_points, 4), np.float32)
    blob[:, :3] = rng.uniform(0.01, 0.09, size=(dense_points, 3)).astype(np.float32)
    blob[:, 3] = rng.uniform(0, 255, size=dense_points).astype(np.float32)
    blob[::3, :3] = 0.0   # and a third of them exactly at the origin
    x = np.concatenate([x, blob])[rng.permutation(len(x) + dense_points)]
    with CloudMerger(max_batch_points=len(x)) as cm:
        out = _voxel_only(cm, x, 0.1, 2)
    o = oracle.voxelgrid(x, [0.1] * 3, 2, True, force64=True)
    st = out["stats"]
    assert st.device_error == 0 and st.voxels_out == o["n"]
    assert (out["voxel_idx"].astype(np.int64) == o["idx"]).all() and (out["voxel_count"] == o["count"]).all()
    assert out["voxel_count"].max() >= dense_points
    assert_bit_equal(out["voxel_xyzi"], o["centroid"], "centroids vs the float oracle (ascending index order)")
    assert st.gpu_ms < 30.0, "the giant voxel must not serialise the launch (%.1f ms)" % st.gpu_ms


@pytest.mark.parametrize("leaf", [0.01, 0.02])
def test_sort_64bit_big_tile_at_size(gpu_ok, oracle, leaf):
    """k_onesweep_pass<unsigned long long, 8> (64-bit keys, the big tile: handle capacity above 1 363 968 keys) on
    2.5 Mi points whose grid exceeds PCL's INT32 cell limit (36 / 39 key bits, 5 passes): membership, counts, order,
    centroids against the 64-bit oracle."""
    n = 5 << 19
    x = synth.uniform_cloud(61, n, extent=(200.0, 200.0, 10.0))
    x[:200000] = synth.uniform_cloud(62, 200000, extent=(3.0, 3.0, 1.0))  # a dense clump: runs that cross tiles
    with CloudMerger(max_batch_points=n) as cm:
        out = _voxel_only(cm, x, leaf, 1)
    o = oracle.voxelgrid(x, [leaf] * 3, 1, True, force64=True)
    o.update(n_voxels=o["n"], n_survivors=n)
    assert out["key_bytes"] == 8 and out["stats"].key_bits > 32 and out["stats"].sort_passes >= 5
    assert out["stats"].pcl_overflow == 1 and o["pcl_overflow"]
    assert check_voxels(out, out["frames"], [o]) <= 1e-5


def test_cfg1_batch_of_64_frames_at_size(gpu_ok, oracle):
    """BASELINE config 1 (2 x 64k points, z-only PassThrough -> unbounded grid) as a 64-frame device batch: the key plan is
    made on the device; every frame against the oracle."""
    c = synth.CONFIGS["cfg1"]
    F, S = 64, c["sensors"]
    n = c["rings"] * c["azimuth"]
    with CloudMerger(max_sensors=S, max_batch_points=F * S * n, max_batch_frames=F) as cm:
        for s in range(S):
            cm.set_extrinsic(s, synth.extrinsic(s, S))
        cm.set_crop(c["passes"])
        cm.set_voxel(c["leaf"], c["min_points"], True)
        frames = [[(synth.lidar_cloud(1000, s, f, c["rings"], c["azimuth"]), 1) for s in range(S)] for f in range(F)]
        segs, per_frame = upload_segments(cm, frames, lambda f, s: LAYOUTS["packed16"])
        cm.run_batch(segs)
        out = cm.fetch_batch_outputs()
    assert out["stats"].frames == F and out["stats"].device_error == 0 and out["stats"].survivors > 1363968
    # frame-segmented: the 6 frame bits are not sorted -- 32-bit records and 4 passes where (frame, index) took 64 bits and 5
    assert out["stats"].key_bytes == 4 and out["stats"].sort_passes == 4 and out["stats"].key_bits == out["key_idx_bits"]
    o = _oracle_frames(oracle, per_frame, c["passes"], [c["leaf"]] * 3, c["min_points"])
    check_survivors(out, out["frames"], o)
    assert check_voxels(out, out["frames"], o) <= 1e-5


def _ragged_batch(cm, oracle, sizes, passes, leaf, min_points, extent, same_cloud=False, seed=7000):
    """A one-sensor device batch whose frames hold sizes[f] points; returns (outputs, oracle frames)."""
    cm.set_extrinsic(0, synth.extrinsic(0, 1))
    cm.set_crop(passes)
    cm.set_voxel(leaf, min_points, True)
    frames = [[(synth.uniform_cloud(seed if same_cloud else seed + f, n, extent=extent)[:n], 1)] for f, n in enumerate(sizes)]
    segs, per_frame = upload_segments(cm, frames, lambda f, s: LAYOUTS["packed16"])
    cm.run_batch(segs)
    out = cm.fetch_batch_outputs()
    return out, _oracle_frames(oracle, per_frame, passes, [leaf] * 3, min_points)


@pytest.mark.parametrize("min_points", [1, 2, 3])
def test_frame_segmented_sort_ragged_frames(gpu_ok, oracle, min_points):
    """Batches of several frames on an unbounded grid sort the bare voxel index, every frame as a segment of its own
    (SortInfo.segmented; 32-bit records, no frame bits): frames that are empty, hold one point, exactly one radix tile, one
    more than a tile, several tiles, and frames whose points the crop removes entirely -- small sort tile (1536 keys)."""
    sizes = [0, 1, 5, 1536, 1537, 0, 9000, 3072, 2, 4607, 4608, 4609, 0, 0, 700, 12000, 1]
    z_only = [(2, -1.5, 1.5, 0)]
    with CloudMerger(max_sensors=1, max_batch_points=sum(sizes), max_batch_frames=len(sizes)) as cm:
        out, o = _ragged_batch(cm, oracle, sizes, z_only, 0.25, min_points, (30.0, 30.0, 4.0))
    st = out["stats"]
    assert st.device_error == 0 and st.frames == len(sizes) and st.key_bytes == 4
    assert st.key_bits == out["key_idx_bits"], "no frame bits were sorted"
    check_survivors(out, out["frames"], o)
    assert check_voxels(out, out["frames"], o) <= 1e-5


def test_frame_segmented_sort_same_cells_in_adjacent_frames(gpu_ok, oracle):
    """Every frame holds the SAME cloud: the last voxel of a frame and the first of the next differ only by the frame, and
    equal indices meet at every frame boundary of the sorted array -- runs must end there. 300 frames (frame starts read from
    global memory past 256), all points kept (no crop window cuts), min_points 2."""
    sizes = [2500] * 300
    z_only = [(2, -100.0, 100.0, 0)]
    with CloudMerger(max_sensors=1, max_batch_points=sum(sizes), max_batch_frames=len(sizes)) as cm:
        out, o = _ragged_batch(cm, oracle, sizes, z_only, 0.5, 2, (12.0, 12.0, 3.0), same_cloud=True)
    st = out["stats"]
    assert st.device_error == 0 and st.key_bytes == 4 and st.key_bits == out["key_idx_bits"]
    assert all(fo["n_voxels"] == o[0]["n_voxels"] for fo in o)
    check_survivors(out, out["frames"], o)
    assert check_voxels(out, out["frames"], o) <= 1e-5


def test_frame_segmented_sort_more_frames_than_threads(gpu_ok, oracle):
    """1500 small frames of 0..600 points: more frames than k_grid_setup has threads (its frame loops run twice), more than
    the centroid pass stages in shared memory, most radix tiles partial."""
    rng = np.random.default_rng(77)
    sizes = [int(v) for v in rng.integers(0, 601, size=1500)]
    z_only = [(2, -1.5, 1.5, 0)]
    with CloudMerger(max_sensors=1, max_batch_points=sum(sizes), max_batch_frames=len(sizes)) as cm:
        out, o = _ragged_batch(cm, oracle, sizes, z_only, 0.3, 2, (20.0, 20.0, 4.0))
    st = out["stats"]
    assert st.device_error == 0 and st.frames == len(sizes) and st.key_bytes == 4 and st.key_bits == out["key_idx_bits"]
    check_survivors(out, out["frames"], o)
    assert check_voxels(out, out["frames"], o) <= 1e-5


def test_frame_segmented_sort_big_tile_and_bounded_plan(gpu_ok, oracle):
    """(i) the big sort tile (capacity above 1 363 968 keys) with frames of unequal size; (ii) a crop BOX whose grid needs
    31 index bits: with the frame bits the key would not fit 32 bits, so the host plans a segmented run (32-bit records,
    4 passes) instead of 64-bit keys."""
    sizes = [400000, 1, 310000, 0, 520000, 250001]
    z_only = [(2, -1.5, 1.5, 0)]
    with CloudMerger(max_sensors=1, max_batch_points=sum(sizes), max_batch_frames=len(sizes)) as cm:
        out, o = _ragged_batch(cm, oracle, sizes, z_only, 0.1, 2, (150.0, 150.0, 4.0))
    st = out["stats"]
    assert st.device_error == 0 and st.key_bytes == 4 and st.key_bits == out["key_idx_bits"] and st.survivors > 400000
    check_survivors(out, out["frames"], o)
    assert check_voxels(out, out["frames"], o) <= 1e-5
    sizes = [60000, 80000, 0, 70000, 50000]
    box = [(2, -1.0, 1.0, 0), (1, -60.0, 60.0, 0), (0, -60.0, 60.0, 0)]       # 0.02 m: 6001 x 6001 x 101 cells: 32 bits
    with CloudMerger(max_sensors=1, max_batch_points=sum(sizes), max_batch_frames=len(sizes)) as cm:
        out, o = _ragged_batch(cm, oracle, sizes, box, 0.02, 1, (100.0, 100.0, 3.0))
    st = out["stats"]
    assert st.device_error == 0 and st.key_bytes == 4 and st.sort_passes == 4 and st.key_bits == out["key_idx_bits"]
    check_survivors(out, out["frames"], o)
    assert check_voxels(out, out["frames"], o) <= 1e-5


def test_cfg3_full_size_host_path_and_batch(gpu_ok, oracle):
    """BASELINE config 3 (8 sensors x 256k points, ROI box, leaf 0.05) at full size: one frame through the host path
    (cm_submit_cloud x 8 + cm_merge_frame) and a 16-frame device batch (the bench shape), every frame against the oracle."""
    c = synth.CONFIGS["cfg3"]
    F, S = 16, c["sensors"]
    n = c["rings"] * c["azimuth"]
    mats = [synth.extrinsic(s, S) for s in range(S)]
    frames = [[(synth.lidar_cloud(3000, s, f, c["rings"], c["azimuth"]), 1) for s in range(S)] for f in range(F)]
    with CloudMerger(max_sensors=S, max_points_per_sensor=n, max_point_step=16, max_batch_points=F * S * n,
                     max_batch_frames=F) as cm:
        for s in range(S):
            cm.set_extrinsic(s, mats[s])
        cm.set_crop(c["passes"])
        cm.set_voxel(c["leaf"], c["min_points"], True)
        for s in range(S):
            cm.submit_cloud(s, frames[0][s][0], n, make_layout(), stamp=s)
        r = cm.merge_frame(capacity=S * n)
        segs, per_frame = upload_segments(cm, frames, lambda f, s: LAYOUTS["packed16"])
        cm.run_batch(segs)
        out = cm.fetch_batch_outputs()
    o = _oracle_frames(oracle, per_frame, c["passes"], [c["leaf"]] * 3, c["min_points"])
    assert (r.survivor_src == o[0]["survivor_src"]).all() and len(r.voxel_idx) == o[0]["n_voxels"] > 10000
    assert_bit_equal(r.survivor_xyzi, o[0]["survivor_xyzi"], "host path survivors")
    assert (r.voxel_idx.astype(np.int64) == o[0]["idx"]).all() and (r.voxel_count == o[0]["count"]).all()
    assert_bit_equal(r.voxel_xyzi, o[0]["centroid"], "host path centroids")
    assert out["stats"].frames == F and out["stats"].points_in == F * S * n and out["key_bytes"] == 4
    check_survivors(out, out["frames"], o)
    assert check_voxels(out, out["frames"], o) <= 1e-5


@pytest.mark.parametrize("leaf,min_points", [(0.05, 1), (1.0, 2)])
def test_cfg5_leaf_sweep_at_16mi_points(gpu_ok, oracle, leaf, min_points):
    """BASELINE config 5 at its full 16 Mi points: the fine end (0.05 m: 8e9 cells, 64-bit keys, beyond PCL's INT32 limit,
    nearly every point alone in its voxel) and the coarse end (1.0 m: 400 k voxels of ~42 points)."""
    n = 1 << 24
    x = synth.uniform_cloud(5000, n)
    with CloudMerger(max_batch_points=n) as cm:
        out = _voxel_only(cm, x, leaf, min_points)
    o = oracle.voxelgrid(x, [leaf] * 3, min_points, True, force64=True)
    o.update(n_voxels=o["n"], n_survivors=n)
    assert out["stats"].pcl_overflow == int(o["pcl_overflow"])
    assert out["key_bytes"] == (4 if out["stats"].key_bits <= 32 else 8)
    assert check_voxels(out, out["frames"], [o]) <= 1e-5


def test_submit_policy_and_unmasked_submissions(gpu_ok, oracle):
    """Latest-wins (my_cloud_fusion's add_*_velodyne) against first-wins (pcl_preprocessing's flag gate,
    pc_preprocessing_main.cpp:330); a cloud submitted for a sensor outside the merge mask ends with that merge instead of
    resurfacing frames_in_flight frames later; a single re-submission after a coalesced multi-submit replaces only its sensor."""
    from cloud_merger_b200 import host_alloc
    S, n = 3, 6000
    mats = [synth.extrinsic(s, S) for s in range(S)]
    a = [synth.lidar_cloud(91, s, 0, 8, n // 8) for s in range(S)]
    b = [synth.lidar_cloud(91, s, 1, 8, n // 8) for s in range(S)]

    def expect(clouds, sensors):
        return oracle.merge_frame([cloud_dict(clouds[s], mats[s][:3]) for s in sensors], synth.ROI_BOX, [0.2] * 3, 1, True, True)

    def same(r, o):
        assert (r.survivor_src == o["survivor_src"]).all()
        assert_bit_equal(r.survivor_xyzi, o["survivor_xyzi"], "survivors")
        assert (r.voxel_idx.astype(np.int64) == o["idx"]).all() and (r.voxel_count == o["count"]).all()
        assert_bit_equal(r.voxel_xyzi, o["centroid"], "centroids")

    for first_wins in (False, True):
        with CloudMerger(max_sensors=S, max_points_per_sensor=n, frames_in_flight=2) as cm:
            for s in range(S):
                cm.set_extrinsic(s, mats[s])
            cm.set_crop(synth.ROI_BOX)
            cm.set_voxel(0.2, 1, True)
            cm.set_submit_policy(first_wins)
            for s in range(S):
                cm.submit_cloud(s, a[s], n, make_layout(), stamp=1)
            cm.submit_cloud(1, b[1], n, make_layout(), stamp=2)      # sensor 1 delivers again before the merge
            r = cm.merge_frame(capacity=S * n)
            mixed = [a[0], a[1] if first_wins else b[1], a[2]]
            same(r, expect(mixed, range(S)))
            assert r.stamp == (1 if first_wins else 2)
            # sensor 2 submitted but masked out: merged frame has sensors 0, 1 only; the cloud of sensor 2 is gone afterwards
            for s in range(S):
                cm.submit_cloud(s, b[s], n, make_layout(), stamp=3)
            r = cm.merge_frame(capacity=S * n, sensor_mask=0b011)
            assert r.used_mask == 0b011
            same(r, expect(b, (0, 1)))
            for _ in range(2):   # both slots come round: nothing stale may surface
                cm.submit_cloud(0, a[0], n, make_layout(), stamp=4)
                r = cm.merge_frame(capacity=S * n)
                assert r.used_mask == 0b001
                same(r, expect(a, (0,)))
    # coalesced multi-submit (one PCIe copy into the frame arena), then sensor 1 alone again: only sensor 1 changes
    arena, addr = host_alloc(S * n * 16)
    for s in range(S):
        arena[s * n * 16:(s + 1) * n * 16] = a[s].view(np.uint8).reshape(-1)
    with CloudMerger(max_sensors=S, max_points_per_sensor=n, frames_in_flight=2) as cm:
        for s in range(S):
            cm.set_extrinsic(s, mats[s])
        cm.set_crop(synth.ROI_BOX)
        cm.set_voxel(0.2, 1, True)
        for rep in range(3):
            cm.submit_clouds_pinned(list(range(S)), [addr + s * n * 16 for s in range(S)], [n] * S, [make_layout()] * S)
            if rep:
                cm.submit_cloud(1, b[1][:n - 7 * rep], n - 7 * rep, make_layout())
            r = cm.merge_frame(capacity=S * n)
            same(r, expect([a[0], b[1][:n - 7 * rep] if rep else a[1], a[2]], range(S)))


def test_concurrent_handles_sorting_on_one_device(gpu_ok, oracle):
    """Six handles run their radix passes at the same time on six streams of one GPU (the node's per-sensor lanes): the
    scanner role of a pass goes to the first CTAs to ARRIVE, so co-scheduled passes neither starve their scanners nor trip
    the (wall-clock) watchdog. Every run must reproduce the handle's own serial result, and one of them the oracle's."""
    import threading
    H, n, rounds = 6, 1500000, 6
    clouds = [synth.uniform_cloud(300 + k, n, extent=(150.0 + 10 * k, 150.0, 8.0)) for k in range(H)]
    leaf = 0.25
    handles = [CloudMerger(max_batch_points=n) for _ in range(H)]
    try:
        bufs, streams, want = [], [], []
        for k, cm in enumerate(handles):
            cm.set_voxel(leaf, 1, True)
            bufs.append(cm.upload(clouds[k]))
            streams.append(cm.stream_create())
            cm.dev_voxelgrid(bufs[k].ptr, n, stream=streams[k])
            o = cm.fetch_batch_outputs(want_sorted=False)
            want.append((o["voxel_idx"].copy(), o["voxel_count"].copy(), o["voxel_xyzi"].copy()))
        oref = oracle.voxelgrid(clouds[0], [leaf] * 3, 1, True, force64=True)
        assert (want[0][0].astype(np.int64) == oref["idx"]).all() and (want[0][1] == oref["count"]).all()
        assert_bit_equal(want[0][2], oref["centroid"], "serial run vs oracle")
        errs = []

        def lane(k):
            try:
                cm = handles[k]
                for _ in range(rounds):
                    cm.dev_voxelgrid(bufs[k].ptr, n, stream=streams[k])
                    st = cm.stats()
                    assert st.device_error == 0
                o = cm.fetch_batch_outputs(want_sorted=False)
                assert (o["voxel_idx"] == want[k][0]).all() and (o["voxel_count"] == want[k][1]).all()
                assert_bit_equal(o["voxel_xyzi"], want[k][2], "handle %d" % k)
            except Exception as e:  # noqa: BLE001
                errs.append((k, e))
        th = [threading.Thread(target=lane, args=(k,)) for k in range(H)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        assert not errs, errs
    finally:
        for cm in handles:
            cm.close()


def test_unbounded_crop_host_path_is_asynchronous_and_graph_replayed(gpu_ok, oracle):
    """A crop that does not bound x, y, z (BASELINE config 1: PassThrough z only) leaves the key width to the device: the host
    enqueues both key widths and never waits in the middle of the frame, so such frames pipeline (merge_async returns before the
    GPU is done) and replay as CUDA graphs like bounded ones. Frames alternate between a 32-bit and a 64-bit grid."""
    S, rings, az = 2, 32, 256
    n = rings * az
    with CloudMerger(max_sensors=S, max_points_per_sensor=n, frames_in_flight=3) as cm:
        mats = [synth.extrinsic(s, S) for s in range(S)]
        for s in range(S):
            cm.set_extrinsic(s, mats[s])
        cm.set_crop([(2, -0.5, 3.0, 0)])
        for leaf, want_bytes in ((0.1, 4), (0.002, 8), (0.1, 4)):
            cm.set_voxel(leaf, 1, True)
            tickets, expect = [], []
            for f in range(3):
                clouds = [synth.lidar_cloud(640, s, f, rings, az) for s in range(S)]
                for s in range(S):
                    cm.submit_cloud(s, clouds[s], n, make_layout(), stamp=f)
                tickets.append(cm.merge_frame_async())
                expect.append(oracle.merge_frame([cloud_dict(c, m[:3]) for c, m in zip(clouds, mats)], [(2, -0.5, 3.0, 0)],
                                                 [leaf] * 3, 1, True, True))
            for f in range(3):
                r = cm.wait_frame(tickets[f], capacity=S * n)
                o = expect[f]
                assert (r.survivor_src == o["survivor_src"]).all()
                assert (r.voxel_idx.astype(np.int64) == o["idx"]).all() and (r.voxel_count == o["count"]).all(), (leaf, f)
                assert_bit_equal(r.voxel_xyzi, o["centroid"], "leaf %g frame %d" % (leaf, f))
                assert cm.stats().key_bytes == want_bytes


def test_wait_frame_view_is_the_same_result_without_a_copy(gpu_ok, oracle):
    """cm_wait_frame_view: pointers into the frame's page-locked result mirrors (written by the frame's own stream) instead of
    copies into caller buffers; three frames in flight, both record layouts."""
    S, n = 3, 5000
    for step in (16, 32):
        with CloudMerger(max_sensors=S, max_points_per_sensor=n, frames_in_flight=3, out_point_step=step) as cm:
            mats = [synth.extrinsic(s, S) for s in range(S)]
            for s in range(S):
                cm.set_extrinsic(s, mats[s])
            cm.set_crop(synth.ROI_BOX)
            cm.set_voxel(0.2, 1, True)
            tickets, expect = [], []
            for f in range(3):
                clouds = [synth.lidar_cloud(66, s, f, 10, n // 10) for s in range(S)]
                for s in range(S):
                    cm.submit_cloud(s, clouds[s], n, make_layout(), stamp=10 + f)
                tickets.append(cm.merge_frame_async())
                expect.append(oracle.merge_frame([cloud_dict(c, m[:3]) for c, m in zip(clouds, mats)], synth.ROI_BOX, [0.2] * 3, 1, True, True))
            for f in range(3):
                v = cm.wait_frame_view(tickets[f])
                a = cm.view_arrays(v)
                o = expect[f]
                assert v.n_voxels == o["n_voxels"] > 50 and v.n_survivors == o["n_survivors"] and v.stamp == 10 + f and v.used_mask == 0b111
                assert (a["voxel_idx"].astype(np.int64) == o["idx"]).all() and (a["voxel_count"] == o["count"]).all()
                rec = a["voxel_xyzi"]
                xyzi = rec if step == 16 else np.concatenate([rec[:, 0:3], rec[:, 4:5]], axis=1)
                assert_bit_equal(xyzi, o["centroid"], "frame %d (view, %d-byte records)" % (f, step))
                if step == 32:
                    assert (rec[:, 3] == 1.0).all()


@pytest.mark.parametrize("leaf,box", [(0.05, [(0, 3.0, 4.5, 0), (1, -1.0, 0.25, 0), (2, -0.5, 3.0, 0)]),      # ~1 % of the points survive
                                      (0.035, [(2, -2.25, 7.1, 0), (0, -33.3, 41.7, 0), (1, -17.9, 12.2, 0)]),  # box not aligned to the leaf, 32 key bits
                                      (0.25, [(0, -60.0, 60.0, 0), (1, -60.0, 60.0, 0), (2, -60.0, 60.0, 0), (3, 20.0, 230.0, 0)])])
def test_keys_from_the_crop_box_grid(gpu_ok, oracle, leaf, box):
    """When the crop is a box that bounds x, y, z, K1 keys the survivors against the BOX's voxel grid and radix pass 0 reads
    the keys through the K1 tile records; the voxel index handed out is re-based on each frame's data-derived grid. Checked
    against the oracle (which follows PCL: grid from the data) for a crop that keeps ~1 % of the points (a radix tile then
    spans hundreds of K1 tiles: the binary-search path), a box that is not aligned to the leaf with a 32-bit key, and an
    intensity window on top of the box; five frames of different sizes, 2.3 M points (the 4096-point K1 tile, the big radix tile)."""
    F, S = 5, 3
    frames = [[(synth.lidar_cloud(900 + f, s, f, 128, 1100 + 97 * f + 13 * s), 1) for s in range(S)] for f in range(F)]
    total = sum(len(p) for fr in frames for p, _ in fr)
    assert total > (1 << 21)
    with CloudMerger(max_sensors=S, max_batch_points=total, max_batch_frames=F) as cm:
        for s in range(S):
            cm.set_extrinsic(s, synth.extrinsic(s, S))
        cm.set_crop(box)
        cm.set_voxel(leaf, 1, True)
        segs, per_frame = upload_segments(cm, frames, lambda f, s: LAYOUTS["packed16" if s != 1 else "pcl32"])
        cm.run_batch(segs)
        out = cm.fetch_batch_outputs()
    o = _oracle_frames(oracle, per_frame, box, [leaf] * 3, 1)
    assert out["key_bytes"] == 4 and out["stats"].device_error == 0
    if leaf == 0.035:
        assert out["stats"].key_bits == 32
    check_survivors(out, out["frames"], o)
    assert check_voxels(out, out["frames"], o) <= 1e-5
    assert sum(fo["n_voxels"] for fo in o) > 1000
