"""Fused-key runs whose crop-box grid has more than 2^(8k) cells sort every frame as a segment of its own (the frame bits stay
in the keys, unranked) with a top digit of up to 384 bins: three radix passes where the bit-based plan took four. Bit-exact
against the oracle at the cell-count edges of the plan (2^24 + 1, 384 * 2^16 and one cell more), with the top digit at
exactly 383, with empty, one-point and exactly-one-tile frames, with 2, 16 and 32 frames, with a sparse crop, in both sort
tile sizes, and through the host path with its captured and replayed graph."""
import numpy as np
import pytest

import edge_inputs as E
from cloud_merger_b200 import CloudMerger, make_layout
from helpers import assert_bit_equal, check_survivors, check_voxels, cloud_dict, upload_segments

pytestmark = pytest.mark.gpu

PACKED = (16, 0, 4, 8, 12)
IDENTITY = np.eye(4)
DIV_2P24_PLUS = (673, 257, 97)      # 2^24 + 1 cells: top digit 256 -> 3 passes
DIV_384_2P16 = (2048, 1024, 12)     # 384 * 2^16 cells: the last cell has top digit 383 -> 3 passes
DIV_384_2P16_PLUS = (1006633, 25, 1)  # 384 * 2^16 + 1 cells: 385 top digits -> 4 passes
SMALL_TILE = 384 * 4                # radix tile of a batch of at most ~1.4 M points


def _box(div):
    return [(a, 0.0, float(div[a]) - 0.5, 0) for a in range(3)]


def _run(frames_xyz, div, crop=None):
    crop = crop or _box(div)
    frames = [[(x, 1)] for x in frames_xyz]
    total = max(1, sum(len(x) for x in frames_xyz))
    with CloudMerger(max_sensors=1, max_batch_points=total, max_batch_frames=len(frames)) as cm:
        cm.set_extrinsic(0, E.identity_extrinsic((0, 0, 0)))
        cm.set_crop(crop)
        cm.set_voxel(1.0, 1, True)
        segs, per_frame = upload_segments(cm, frames, lambda f, s: PACKED)
        cm.run_batch(segs)
        out = cm.fetch_batch_outputs()
    return out, per_frame, crop


def _check(oracle, out, per_frame, crop, passes, div):
    o = [oracle.merge_frame(cds, crop, [1.0] * 3, 1, True, True) for cds in per_frame]
    st = out["stats"]
    idx_bits = E.bits_for(int(np.prod(np.asarray(div, np.int64))))
    assert st.device_error == 0 and st.key_bytes == 4 and out["key_idx_bits"] == idx_bits
    assert st.key_bits == idx_bits + E.bits_for(len(per_frame))     # the key width keeps its frame bits
    assert st.sort_passes == passes
    check_survivors(out, out["frames"], o)
    check_voxels(out, out["frames"], o)
    return o


@pytest.mark.parametrize("div,F,passes", [(DIV_2P24_PLUS, 2, 3), (DIV_384_2P16, 2, 3), (DIV_384_2P16_PLUS, 2, 4),
                                          (DIV_2P24_PLUS, 16, 3), (DIV_2P24_PLUS, 32, 3), (DIV_384_2P16, 1, 3)])
def test_cell_count_edges(gpu_ok, oracle, div, F, passes):
    xs = [E.grid_cloud(900 + f, div, n_filler=6000 + 37 * f) for f in range(F)]
    out, per_frame, crop = _run(xs, div)
    o = _check(oracle, out, per_frame, crop, passes, div)
    if div == DIV_384_2P16:   # the corner cell C - 1 is occupied: its top digit is 383, the last bin of the wide pass
        cells = int(np.prod(np.asarray(div, np.int64)))
        assert ((cells - 1) >> 16) == 383 and any(int(fo["idx"].max()) >> 16 == 383 for fo in o)


@pytest.mark.parametrize("big", [False, True])
def test_empty_one_point_and_one_tile_frames(gpu_ok, oracle, big):
    """Frames of 0, 1 and exactly one radix tile of points between ordinary ones; big: enough points for the large sort tile."""
    base = E.grid_cloud(31, DIV_2P24_PLUS, n_filler=(800000 if big else 20000))
    one = base[:1].copy()
    tile = E.grid_cloud(32, DIV_2P24_PLUS, n_filler=SMALL_TILE - 8)
    assert len(tile) == SMALL_TILE
    empty = np.zeros((0, 4), np.float32)
    xs = [base, empty, one, tile, E.grid_cloud(33, DIV_2P24_PLUS, n_filler=(700000 if big else 9000)), empty]
    out, per_frame, crop = _run(xs, DIV_2P24_PLUS)
    _check(oracle, out, per_frame, crop, 3, DIV_2P24_PLUS)


def test_sparse_crop(gpu_ok, oracle):
    """A crop that keeps about 2 % of the points: a radix tile spans more than 32 K1 tiles (pass 0's binary search)."""
    rng = np.random.default_rng(5)
    xs = []
    for f in range(3):
        inside = E.grid_cloud(40 + f, DIV_2P24_PLUS, n_filler=8000)
        outside = np.empty((400000, 4), np.float32)
        outside[:, 0] = rng.uniform(1000.0, 60000.0, len(outside))
        outside[:, 1] = rng.uniform(0.5, 256.5, len(outside))
        outside[:, 2] = rng.uniform(0.5, 96.5, len(outside))
        outside[:, 3] = rng.uniform(0, 255, len(outside))
        x = np.concatenate([inside, outside])
        xs.append(x[rng.permutation(len(x))])
    out, per_frame, crop = _run(xs, DIV_2P24_PLUS)
    _check(oracle, out, per_frame, crop, 3, DIV_2P24_PLUS)
    assert out["stats"].survivors < 0.03 * out["stats"].points_in


def test_single_frame_host_path_captured_replayed(gpu_ok, oracle):
    """One frame through cm_merge_frame: plain enqueue, graph capture, replay -- a single frame is sorted as one segment."""
    div = DIV_384_2P16
    crop = _box(div)
    clouds = [E.grid_cloud(70 + f, div, n_filler=30000) for f in range(3)]
    n = max(len(x) for x in clouds)
    with CloudMerger(max_sensors=1, max_points_per_sensor=n, frames_in_flight=1) as cm:
        cm.set_extrinsic(0, IDENTITY)
        cm.set_crop(crop)
        cm.set_voxel(1.0, 1, True)
        for f, x in enumerate(clouds):
            cm.submit_cloud(0, x, len(x), make_layout())
            r = cm.merge_frame(capacity=n)
            assert cm.stats().sort_passes == 3, f
            o = oracle.merge_frame([cloud_dict(x, IDENTITY)], crop, [1.0] * 3, 1, True, True)
            assert (r.survivor_src == o["survivor_src"]).all(), f
            assert (r.voxel_idx.astype(np.int64) == o["idx"]).all() and (r.voxel_count == o["count"]).all(), f
            assert_bit_equal(r.voxel_xyzi, o["centroid"], "frame %d centroids" % f)
