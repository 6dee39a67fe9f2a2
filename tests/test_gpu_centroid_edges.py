"""GPU parity of the centroid pass at its tile, run-length and hand-over edges (-m gpu): the run-layout clouds of
tests/edge_inputs.py (family R) through every instantiation of k_voxel_centroid and every emit path of it and of
finish_tail_run -- 32-bit record keys, 64-bit key arrays, the sentinel frame of non-finite points, frame-segmented batches
(frame starts in shared memory and in global memory), sorted frame bits, K1's fused crop-box keys, the 32-byte PCL record,
downsample_all off, the host path with its captured and replayed graph, and the epoch wrap-around of the look-back words.
Every case asserts the stats that show which path ran, and matches the float oracle bit for bit (ids, order, counts,
centroids, membership, per-frame voxel ranges) and the float64 oracle within the derived float32 bound."""
import numpy as np
import pytest

import edge_inputs as E
from cloud_merger_b200 import CloudMerger, CloudMergerError, _lib, make_layout
from helpers import assert_bit_equal, assert_centroids_within_bound, check_survivors, check_voxels, cloud_dict, upload_segments

pytestmark = pytest.mark.gpu

F32 = np.float32
PACKED = (16, 0, 4, 8, 12)
Z_ONLY = [(2, -1e6, 1e6, 0)]     # crops nothing and bounds no grid: the batch plans its sort on the device
IDENTITY = E.identity_extrinsic((0, 0, 0))


def _cloud(name, n_nonfinite=0, far=False, seed=None):
    runs, _ = E.layout(name, seed=7)
    return E.run_layout_cloud(runs, seed=len(name) if seed is None else seed, n_nonfinite=n_nonfinite, far=far)


def _dev_voxelgrid(x, min_points, is_dense=True, downsample_all=True, out_point_step=16):
    with CloudMerger(max_batch_points=len(x), out_point_step=out_point_step) as cm:
        cm.set_voxel(1.0, min_points, downsample_all)
        buf = cm.upload(x)
        cm.dev_voxelgrid(buf.ptr, len(x), is_dense=is_dense)
        return cm.fetch_batch_outputs()


def _check_single(out, x, min_points, is_dense=True, downsample_all=True):
    """One frame against the oracle: bit-exact voxels, the float64 bound, voxels_out, no device error."""
    o = _oracle_voxelgrid(x, min_points, is_dense, downsample_all)
    st = out["stats"]
    assert st.device_error == 0 and st.frames == 1
    assert st.voxels_out == o["n"], (st.voxels_out, o["n"])
    check_voxels(out, out["frames"], [o], check_membership=is_dense)
    assert_centroids_within_bound(out["voxel_xyzi"], o["centroid_f64"], x, o["point_idx"], o["idx"], o["count"])
    return o


def _oracle_voxelgrid(x, min_points, is_dense=True, downsample_all=True):
    from oracle import cm_oracle_py
    o = cm_oracle_py.voxelgrid(x, [1.0] * 3, min_points, downsample_all, force64=True, is_dense=is_dense)
    o.update(n_voxels=o["n"], n_survivors=len(x))
    return o


def _cells_bits(o):
    return E.bits_for(int(np.prod(o["div_b"].astype(np.int64))))


# ---- k_voxel_centroid<uint32_t>: one dense frame, 32-bit (key, value) records ----------------------------------------------
U32_CASES = ([(n, mp) for n in E.R_LAYOUTS for mp in (1, 2)] + [(n, int(n.split(":")[1])) for n in E.R_MINPTS] +
             [("bounds", 9), ("leave", 25), ("persist", 1), ("persist", 3)])


@pytest.mark.parametrize("name,min_points", U32_CASES)
def test_u32_records(gpu_ok, name, min_points):
    x = _cloud(name)
    out = _dev_voxelgrid(x, min_points)
    o = _check_single(out, x, min_points)
    assert out["key_bytes"] == 4 and out["stats"].key_bits == _cells_bits(o)


# ---- k_voxel_centroid<unsigned long long>: a far corner widens the grid past 32 index bits ---------------------------------
@pytest.mark.parametrize("name,min_points", [("bounds", 2), ("leave", 1), ("leave", 26), ("dense", 1), ("minpts:25:24", 25),
                                             ("end:handover-partial", 1), ("persist", 2)])
def test_u64_arrays_with_far_corner(gpu_ok, name, min_points):
    x = _cloud(name, far=True)
    out = _dev_voxelgrid(x, min_points)
    o = _check_single(out, x, min_points)
    assert out["key_bytes"] == 8 and out["stats"].key_bits == _cells_bits(o) == 33


# ---- the sentinel frame: non-finite rows sort last, behind a finite run that is handed over ---------------------------------
@pytest.mark.parametrize("min_points", [1, 2])
@pytest.mark.parametrize("far", [False, True])
def test_sentinel_frame_after_a_handed_over_run(gpu_ok, min_points, far):
    """5000 non-finite rows (more than two tiles of sentinel keys) right after the last finite run, which leaves its tile by
    300 points and is finished by finish_tail_run: its rounds must stop at the sentinel keys, and no non-finite point is
    ever emitted or counted."""
    rl = E.RunList(5)
    E.leave_block(rl)
    rl.fill(E.next_edge(rl.pos, E.CE_TILE) - 7).run(7 + 300)
    x = E.run_layout_cloud(rl.runs, seed=41, n_nonfinite=5000, far=far)
    out = _dev_voxelgrid(x, min_points, is_dense=False)
    o = _check_single(out, x, min_points, is_dense=False)
    st = out["stats"]
    assert st.key_bits == _cells_bits(o) + 1 and out["key_bytes"] == (8 if far else 4)
    assert int(out["voxel_count"].sum()) == int(o["count"].sum()) <= int(np.isfinite(x[:, :3]).all(axis=1).sum())
    assert (out["voxel_count"] == 307).any(), "the handed-over run before the sentinel keys"


# ---- batches: frame-segmented runs, sorted frame bits, fused crop-box keys ---------------------------------------------------
def _run_batch(frames, passes, min_points, dense=1):
    """run_batch of one sensor cloud per frame against the oracle; membership is checked where every survivor is finite
    (non-finite survivors sort behind all frames, into the sentinel frame)."""
    F = len(frames)
    total = sum(len(x) for x in frames)
    with CloudMerger(max_sensors=1, max_batch_points=max(total, 1), max_batch_frames=F) as cm:
        cm.set_extrinsic(0, IDENTITY)
        cm.set_crop(passes)
        cm.set_voxel(1.0, min_points, True)
        segs, per_frame = upload_segments(cm, [[(x, dense)] for x in frames], lambda f, s: PACKED)
        cm.run_batch(segs)
        out = cm.fetch_batch_outputs()
    o = [_oracle_merge(cds, passes, min_points) for cds in per_frame]
    st = out["stats"]
    assert st.device_error == 0 and st.frames == F
    assert st.voxels_out == sum(fo["n_voxels"] for fo in o)
    check_survivors(out, out["frames"], o)
    check_voxels(out, out["frames"], o, check_membership=bool(dense))
    for f, (fi, fo) in enumerate(zip(out["frames"], o)):
        if fo["n_voxels"]:
            assert_centroids_within_bound(out["voxel_xyzi"][fi.voxel_begin:fi.voxel_end], fo["centroid_f64"],
                                          fo["survivor_xyzi"], fo["point_idx"], fo["idx"], fo["count"], "frame %d" % f)
    return out, o


def _oracle_merge(cds, passes, min_points):
    from oracle import cm_oracle_py
    return cm_oracle_py.merge_frame(cds, passes, [1.0] * 3, min_points, True, True)


def _frame_tail_kinds(runs, cuts):
    w = E.centroid_walk(np.unique(np.r_[0, cuts, np.cumsum(runs)[:-1]]), sum(runs), np.r_[0, cuts])
    return set(np.where(w["straddles"][w["handed"]], "straddles", "one-frame").tolist())


@pytest.mark.parametrize("name", ["seg3", "seg300"])
@pytest.mark.parametrize("min_points", [1, 2, 25])
def test_segmented_batch(gpu_ok, name, min_points):
    """k_voxel_centroid<u64, true>: the records carry the bare voxel index and the frame comes from the position -- from
    shared memory for 3 frames, from global memory for 300. Frame edges at every R-bounds offset, empty frames, the same
    voxel index on both sides of a frame edge inside an inline walk and inside a tail round, and handed-over runs in tiles
    that straddle frames (counted per voxel) and in tiles of one frame (counted per tile)."""
    runs, cuts, _ = E.batch_layout(name, seed=3)
    frames = E.run_layout_frames(runs, cuts, seed=11)
    assert _frame_tail_kinds(runs, cuts) == {"straddles", "one-frame"}
    out, o = _run_batch(frames, Z_ONLY, min_points)
    st = out["stats"]
    assert st.key_bytes == 4 and st.key_bits == out["key_idx_bits"] == max(_cells_bits(fo) for fo in o if fo["n_survivors"])


@pytest.mark.parametrize("name", ["seg3", "seg300"])
def test_frame_bits_sorted(gpu_ok, name):
    """The same batches with non-finite rows and no crop pass: the non-finite survivors need the sentinel frame, so the frame
    bits are sorted with the index (k_voxel_centroid<u64> on 64-bit keys)."""
    runs, cuts, _ = E.batch_layout(name, seed=3)
    frames = E.run_layout_frames(runs, cuts, seed=11, n_nonfinite=3)
    out, o = _run_batch(frames, [], 2, dense=0)
    st = out["stats"]
    idx_bits = max(_cells_bits(fo) for fo in o if fo["n_survivors"])
    assert out["key_idx_bits"] == idx_bits and st.key_bits == idx_bits + E.bits_for(len(frames) + 1) > out["key_idx_bits"]


@pytest.mark.parametrize("min_points", [1, 2])
def test_fused_box_keys(gpu_ok, min_points):
    """K1 keys the survivors on the grid of a crop box that bounds x, y and z; every frame has another data grid (shifted by
    whole cells) and frames 1 and 2 hold handed-over runs: finish_tail_run must re-base each onto its own frame's grid."""
    runs, cuts, _ = E.batch_layout("seg3", seed=3)
    frames = E.run_layout_frames(runs, cuts, seed=11, shift=(3, 2, 1))
    hi = [float(np.nanmax(np.concatenate(frames)[:, a])) + 2.0 for a in range(3)]
    box = [(a, -0.5, hi[a], 0) for a in range(3)]
    out, o = _run_batch(frames, box, min_points)
    st = out["stats"]
    assert [list(fi.min_b) for fi in out["frames"]] == [[0, 0, 0], [3, 2, 1], [6, 4, 2]]
    box_bits = E.bits_for(int(np.prod([int(np.floor(h)) + 2 for h in hi])))   # floor(-0.5) = -1 .. floor(hi)
    assert st.key_bytes == 4 and out["key_idx_bits"] == box_bits and st.key_bits == box_bits + E.bits_for(3)
    assert st.survivors == st.points_in


# ---- output variants: the 32-byte PCL record and downsample_all off, on ordinary and handed-over voxels --------------------
@pytest.mark.parametrize("out_point_step,downsample_all", [(32, True), (32, False), (16, False)])
@pytest.mark.parametrize("far", [False, True])
def test_output_variants(gpu_ok, out_point_step, downsample_all, far):
    x = _cloud("leave", far=far)
    out = _dev_voxelgrid(x, 1, downsample_all=downsample_all, out_point_step=out_point_step)
    o = _check_single(out, x, 1, downsample_all=downsample_all)
    rec = out["voxel_records"]
    assert (out["voxel_count"] > 1000).sum() >= 10   # handed-over voxels among them
    if out_point_step == 32:
        assert_bit_equal(rec[:, 3], np.ones(len(rec), F32), "pad word after z")
        assert_bit_equal(rec[:, 5:8], np.zeros((len(rec), 3), F32), "pad words after the intensity")
    if not downsample_all:
        assert (out["voxel_xyzi"][:, 3].view(np.uint32) == 0).all(), "intensity must be exactly +0.0"
    assert len(rec) == o["n"]


# ---- host path: plain enqueue, CUDA-graph capture, replay --------------------------------------------------------------------
@pytest.mark.parametrize("min_points", [1, 2])
def test_host_path_captured_replayed(gpu_ok, oracle, min_points):
    runs, _ = E.layout("leave", seed=7)
    clouds = [E.run_layout_cloud(runs, seed=60 + f) for f in range(3)]
    n = len(clouds[0])
    with CloudMerger(max_sensors=1, max_points_per_sensor=n, frames_in_flight=1) as cm:
        cm.set_extrinsic(0, IDENTITY)
        cm.set_crop(Z_ONLY)
        cm.set_voxel(1.0, min_points, True)
        for f, x in enumerate(clouds):
            cm.submit_cloud(0, x, len(x), make_layout())
            r = cm.merge_frame(capacity=n)
            o = oracle.merge_frame([cloud_dict(x, IDENTITY)], Z_ONLY, [1.0] * 3, min_points, True, True)
            assert (r.survivor_src == o["survivor_src"]).all(), f
            assert (r.voxel_idx.astype(np.int64) == o["idx"]).all() and (r.voxel_count == o["count"]).all(), f
            assert_bit_equal(r.voxel_xyzi, o["centroid"], "frame %d centroids" % f)
            assert_centroids_within_bound(r.voxel_xyzi, o["centroid_f64"], o["survivor_xyzi"], o["point_idx"], o["idx"],
                                          o["count"], "frame %d" % f)


# ---- the epoch of the look-back words wraps around ------------------------------------------------------------------------
EPOCH_WRAP = 1 << 30
EPOCH_START = EPOCH_WRAP - 64 - 3 * 16   # runs 1-3 below the wrap, run 4 wraps (*epoch + 64 >= 2^30), runs 5-6 after it


def test_epoch_start_is_validated(gpu_ok, monkeypatch):
    for bad in ("8", str(EPOCH_WRAP - 64), str(EPOCH_WRAP), "-16", "16x", ""):
        monkeypatch.setenv("CM_EPOCH_START", bad)
        with pytest.raises(CloudMergerError) as e:
            CloudMerger(max_batch_points=16)
        assert e.value.code == _lib.CM_E_INVALID, bad
    monkeypatch.setenv("CM_EPOCH_START", str(EPOCH_WRAP - 80))
    CloudMerger(max_batch_points=16).close()


def test_epoch_wraps_around(gpu_ok, oracle, monkeypatch):
    """One handle starts its epochs three runs before the wrap-around and alternates an R-leave cloud (dev_voxelgrid) with a
    segmented batch (run_batch) for 6 runs across it: the wrap clears the look-back words of the radix passes and of the
    centroid pass, and every run matches the oracle."""
    monkeypatch.setenv("CM_EPOCH_START", str(EPOCH_START))
    runs, cuts, _ = E.batch_layout("seg3", seed=3)
    frames = E.run_layout_frames(runs, cuts, seed=11)
    lruns, _ = E.layout("leave", seed=7)
    total = max(sum(len(x) for x in frames), sum(lruns))
    with CloudMerger(max_sensors=1, max_batch_points=total, max_batch_frames=len(frames)) as cm:
        monkeypatch.delenv("CM_EPOCH_START")
        cm.set_extrinsic(0, IDENTITY)
        cm.set_crop(Z_ONLY)
        cm.set_voxel(1.0, 2, True)
        segs, per_frame = upload_segments(cm, [[(x, 1)] for x in frames], lambda f, s: PACKED)
        ob = [_oracle_merge(cds, Z_ONLY, 2) for cds in per_frame]
        for run in range(6):
            if run % 2 == 0:
                x = E.run_layout_cloud(lruns, seed=70 + run)
                buf = cm.upload(x)
                cm.dev_voxelgrid(buf.ptr, len(x))
                out = cm.fetch_batch_outputs()
                buf.free()
                o = oracle.voxelgrid(x, [1.0] * 3, 2, True, force64=True)
                o.update(n_voxels=o["n"], n_survivors=len(x))
                assert out["stats"].device_error == 0 and out["stats"].voxels_out == o["n"], run
                check_voxels(out, out["frames"], [o])
            else:
                cm.run_batch(segs)
                out = cm.fetch_batch_outputs()
                st = out["stats"]
                assert st.device_error == 0 and st.key_bits == out["key_idx_bits"], run
                assert st.voxels_out == sum(fo["n_voxels"] for fo in ob), run
                check_survivors(out, out["frames"], ob)
                check_voxels(out, out["frames"], ob)
