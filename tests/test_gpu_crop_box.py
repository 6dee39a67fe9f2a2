"""GPU tests of the pcl::CropBox stages (-m gpu): survivors, their source indices and the voxels of the library against the
float oracle composed as transform -> PassThrough chain -> boxes -> concat -> VoxelGrid (tests/crop_box_cases.py), bit for
bit, through every K1 record layout and chain kind, with and without fused keys, with 1, 2 and 8 boxes, in 1024- and
4096-point tiles, in multi-frame batches, on the host path across graph capture and replay, and at BASELINE config 3 size."""
import numpy as np
import pytest

import crop_box_cases as K
from cloud_merger_b200 import CloudMerger, CloudMergerError, _lib, make_layout, synth
from helpers import assert_bit_equal, check_survivors, check_voxels, cloud_dict, upload_segments

pytestmark = pytest.mark.gpu

LAYOUTS = {"packed16": (16, 0, 4, 8, 12), "pcl32": (32, 0, 4, 8, 16), "velodyne22": (22, 0, 4, 8, 12),
           "livox18": (18, 0, 4, 8, 12)}
CHAINS = {"none": [],
          "box": [(0, -8.0, 8.0, 0), (1, -6.0, 6.0, 0), (2, -3.0, 4.0, 0)],
          "box_i": [(0, -8.0, 8.0, 0), (1, -6.0, 6.0, 0), (2, -3.0, 4.0, 0), (3, 10.0, 240.0, 0)],
          "general": [(2, -3.0, 4.0, 0), (0, -0.5, 0.5, 1)]}
SMALL_NEG = [K.box((-0.25, 1.0, 0.0), (0.25, 1.5, 1.0), negative=True),
             K.box((2.0, -1.75, 0.5), (2.5, -1.25, 1.5), rotation=(0.0, 0.0, 0.3), negative=True)]
SETS = {"1neg": [K.EGO], "1pos": [K.BOXES["rpy_pos"]], "2": [K.BOXES["axis_pos"], K.EGO],
        "8": [K.BOXES["axis_pos"], K.BOXES["tiny_rot_pos"], K.EGO, K.BOXES["axis_neg"], K.BOXES["transform_neg"]] + SMALL_NEG +
             [K.box((-4.0, -2.5, -1.0), (4.5, 2.5, 2.0), rotation=(0.02, 0.0, -0.1))]}
IDENT = np.eye(4, dtype=np.float32)


def _sensor_clouds(seed, boxes, with_nan=True):
    """Sensor 0 (identity extrinsic, so the face points stay on the faces): edge clouds of every box; sensor 1: a small
    lidar cloud through a real extrinsic."""
    edge = np.concatenate([K.edge_cloud(seed + k, b, n_face=8, n_random=600, special=with_nan) for k, b in enumerate(boxes)])
    lidar = synth.lidar_cloud(seed, 1, 0, 16, 256, nan_frac=0.01 if with_nan else 0.0)
    return edge, lidar


def _setup(cm, chain, boxes, leaf=0.1):
    cm.set_extrinsic(0, IDENT)
    cm.set_extrinsic(1, synth.extrinsic(1, 4))
    cm.set_crop(chain)
    cm.set_crop_boxes([K.to_cm(b) for b in boxes])
    cm.set_voxel(leaf, 1, True)


def _check_run(oracle, cm, per_frame, chain, boxes, voxels, leaf=0.1, min_points=1):
    out = cm.fetch_batch_outputs()
    o = [K.merge_expectation(oracle, cds, chain, boxes, leaf, min_points) for cds in per_frame]
    assert out["stats"].device_error == 0
    check_survivors(out, out["frames"], o)
    if voxels:
        fin = all(np.isfinite(f["survivor_xyzi"][:, :3]).all() for f in o)
        check_voxels(out, out["frames"], o, check_membership=fin)
    return out, o


@pytest.mark.parametrize("bset", list(SETS))
@pytest.mark.parametrize("entry", ["run_batch", "transform_crop"])
@pytest.mark.parametrize("chain", list(CHAINS))
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_layouts_chains_and_box_sets(gpu_ok, oracle, layout, chain, entry, bset):
    """One frame of two sensors in 1024-point tiles. run_batch with an x/y/z chain takes the fused-key kernels; the
    transform_crop entry runs the same chain without keys. Non-dense sensor 0 (non-finite rows dropped by the first box
    when no pass runs), dense sensor 1 (NaN rows survive a positive first box without passes)."""
    boxes = SETS[bset]
    edge, lidar = _sensor_clouds(11 + len(bset) + 5 * len(chain), boxes)
    n = len(edge) + len(lidar)
    with CloudMerger(max_sensors=2, max_batch_points=n) as cm:
        _setup(cm, CHAINS[chain], boxes)
        segs, per_frame = upload_segments(cm, [[(edge, 0), (lidar, 1)]], lambda f, s: LAYOUTS[layout])
        if entry == "run_batch":
            cm.run_batch(segs)
        else:
            cm.dev_transform_crop(segs)
        out, o = _check_run(oracle, cm, per_frame, CHAINS[chain], boxes, entry == "run_batch")
    m = o[0]["n_survivors"]
    assert 0 < m < n
    if entry == "run_batch" and chain.startswith("box"):
        assert out["key_bytes"] == 4   # the fused-key path stayed eligible


@pytest.mark.parametrize("chain", ["box", "general"])
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_big_batch_tiles(gpu_ok, oracle, layout, chain):
    """2^21 points: the 4096-point tile kernels (512 threads x 8 items), eight boxes, one BASELINE config 3 frame."""
    boxes = SETS["8"]
    clouds, mats = synth.frame_clouds("cfg3", 77, 0, nan_frac=0.002)
    with CloudMerger(max_sensors=8, max_batch_points=sum(len(c) for c in clouds)) as cm:
        for s in range(8):
            cm.set_extrinsic(s, mats[s])
        cm.set_crop(CHAINS[chain])
        cm.set_crop_boxes([K.to_cm(b) for b in boxes])
        cm.set_voxel(0.1, 1, True)
        segs, per_frame = upload_segments(cm, [[(c, s % 2) for s, c in enumerate(clouds)]], lambda f, s: LAYOUTS[layout])
        cm.run_batch(segs)
        _, o = _check_run(oracle, cm, per_frame, CHAINS[chain], boxes, True)
    assert o[0]["n_survivors"] > 1000


@pytest.mark.parametrize("chain", ["none", "box", "general"])
def test_multi_frame_segmented_batch(gpu_ok, oracle, chain):
    """Three frames of two sensors, mixed layouts and dense flags, boxes applied per segment; frame slices, keys and voxels
    per frame."""
    boxes = SETS["2"]
    frames = []
    for f in range(3):
        edge, lidar = _sensor_clouds(200 + 10 * f, boxes)
        frames.append([(edge, f % 2), (lidar, 1 - f % 2)])
    names = list(LAYOUTS)
    total = sum(len(x) for fr in frames for x, _ in fr)
    with CloudMerger(max_sensors=2, max_batch_points=total, max_batch_frames=3) as cm:
        _setup(cm, CHAINS[chain], boxes)
        segs, per_frame = upload_segments(cm, frames, lambda f, s: LAYOUTS[names[(f + 2 * s) % 4]])
        cm.run_batch(segs)
        _, o = _check_run(oracle, cm, per_frame, CHAINS[chain], boxes, True)
    assert all(fr["n_survivors"] > 0 for fr in o)


def test_host_path_boxes_change_between_frames(gpu_ok, oracle):
    """cm_merge_frame on frames of one shape while the boxes change: A A A (plain, capture, replay) B B B A A. Each frame is
    checked against the oracle with the boxes set for it; the B frames keep a different set of points than A would, so a
    replay of the A graph (a stale stage table) would fail."""
    chain = CHAINS["box"]
    A, B = SETS["1neg"], [K.BOXES["axis_neg"], K.BOXES["rpy_pos"]]
    plan = [A, A, A, B, B, B, A, A]
    n = None
    with CloudMerger(max_sensors=2, max_points_per_sensor=40000, frames_in_flight=1) as cm:
        _setup(cm, chain, A)
        for f, boxes in enumerate(plan):
            cm.set_crop_boxes([K.to_cm(b) for b in boxes])
            edge, lidar = _sensor_clouds(300 + f, A + B, with_nan=False)
            edge, lidar = edge[:12000], lidar[:4000]     # the same shape every frame
            n = n or len(edge) + len(lidar)
            assert len(edge) + len(lidar) == n
            cm.submit_cloud(0, edge, len(edge), make_layout())
            cm.submit_cloud(1, lidar, len(lidar), make_layout())
            r = cm.merge_frame(capacity=n)
            cds = [cloud_dict(edge, IDENT), cloud_dict(lidar, cm.get_extrinsic(1))]
            o = K.merge_expectation(oracle, cds, chain, boxes, 0.1)
            other = K.merge_expectation(oracle, cds, chain, B if boxes is A else A, 0.1)
            assert not np.array_equal(o["survivor_src"], other["survivor_src"])
            assert (r.survivor_src == o["survivor_src"]).all(), f
            assert_bit_equal(r.survivor_xyzi, o["survivor_xyzi"], "frame %d survivors" % f)
            assert (r.voxel_idx.astype(np.int64) == o["idx"]).all() and (r.voxel_count == o["count"]).all(), f
            assert_bit_equal(r.voxel_xyzi, o["centroid"], "frame %d centroids" % f)


def test_cfg3_full_size_ego_box(gpu_ok, oracle):
    """BASELINE config 3 frame (8 sensors x 256k points, ROI box crop, leaf 0.05) with a negative ego box: bit-exact, and
    the fused-key path is still taken."""
    spec = synth.CONFIGS["cfg3"]
    clouds, mats = synth.frame_clouds("cfg3", 3000, 0)
    n = sum(len(c) for c in clouds)
    with CloudMerger(max_sensors=8, max_batch_points=n) as cm:
        for s in range(8):
            cm.set_extrinsic(s, mats[s])
        cm.set_crop(spec["passes"])
        cm.set_crop_boxes([K.to_cm(K.EGO)])
        cm.set_voxel(spec["leaf"], spec["min_points"], True)
        segs, per_frame = upload_segments(cm, [[(c, 1) for c in clouds]], lambda f, s: LAYOUTS["packed16"])
        cm.run_batch(segs)
        out, o = _check_run(oracle, cm, per_frame, spec["passes"], [K.EGO], True, spec["leaf"], spec["min_points"])
    no_box = K.merge_expectation(oracle, per_frame[0], spec["passes"], [], spec["leaf"], spec["min_points"])
    assert o[0]["n_survivors"] < no_box["n_survivors"], "the ego box removes points of the vehicle"
    assert out["key_bytes"] == 4


def test_set_crop_boxes_refusals(gpu_ok):
    with CloudMerger(max_sensors=1, max_batch_points=1024) as cm:
        ok = K.to_cm(K.EGO)
        for bad_n in (-1, _lib.CM_MAX_CROP_BOXES + 1):
            arr = (_lib.CmCropBox * (_lib.CM_MAX_CROP_BOXES + 1))(*([ok] * (_lib.CM_MAX_CROP_BOXES + 1)))
            assert cm._lib.cm_set_crop_boxes(cm._h, bad_n, arr) == _lib.CM_E_INVALID
        for field in ("min", "max"):
            b = K.to_cm(K.EGO)
            getattr(b, field)[1] = float("nan")
            with pytest.raises(CloudMergerError) as e:
                cm.set_crop_boxes([b])
            assert e.value.code == _lib.CM_E_INVALID
        cm.set_crop_boxes([ok] * _lib.CM_MAX_CROP_BOXES)
        cm.set_crop_boxes([])
