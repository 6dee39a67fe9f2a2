"""Shared helpers of the test-suite: input construction and comparisons (tests only)."""
from __future__ import annotations

import json
import os

import numpy as np

from cloud_merger_b200 import make_layout, synth

HERE = os.path.dirname(os.path.abspath(__file__))


def host_function(name, source="cm_api.cu"):
    """The text of the host function `int name(...)` in cloud_merger_b200/csrc/<source>, up to its closing brace."""
    with open(os.path.join(os.path.dirname(HERE), "cloud_merger_b200", "csrc", source)) as f:
        src = f.read()
    a = src.index("\nint %s(" % name) + 1
    return src[a:src.index("\n}\n", a)]


def known_answer():
    with open(os.path.join(HERE, "golden", "known_answer.json")) as f:
        d = json.load(f)

    def arr(rows):
        return np.array([[float("nan") if v == "nan" else float(v) for v in r] for r in rows], np.float32)
    d["A"] = arr(d["sensor_A_xyzi"])
    d["B"] = arr(d["sensor_B_xyzi"])
    return d


def cloud_dict(xyzi, m, is_dense=1, point_step=16, off_x=0, off_y=4, off_z=8, off_i=12):
    """Oracle-side description of one sensor cloud (bytes in the given PointCloud2 layout)."""
    data = synth.pack_cloud(xyzi, point_step, off_x, off_y, off_z, off_i)
    return dict(data=data, n_points=len(xyzi), point_step=point_step, off_x=off_x, off_y=off_y, off_z=off_z,
                off_i=off_i, is_dense=int(is_dense), m=np.asarray(m, np.float32).reshape(-1)[:12].copy())


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_bit_equal(a, b, what=""):
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, a.shape, b.shape)
    same = (bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))
    if not same.all():
        bad = np.argwhere(~same)
        raise AssertionError("%s: %d of %d values differ bitwise, first at %s: %r vs %r" % (
            what, len(bad), a.size, bad[0], a[tuple(bad[0])], b[tuple(bad[0])]))


def rel_err(g, o):
    g = np.asarray(g, np.float64)
    o = np.asarray(o, np.float64)
    return np.abs(g - o) / np.maximum(np.abs(o), 1e-30)


CENTROID_RTOL = 1e-5  # north_star: centroids within 1e-5 relative tolerance


def assert_centroids_close(g, o_f64, what=""):
    """|g - o| <= 1e-5 * max(|o|, tiny) per component, with an absolute floor of 1e-5 * leaf-scale for values that
    cancel to ~0 (a centroid coordinate near 0 has no meaningful relative error)."""
    g = np.asarray(g, np.float64)
    o = np.asarray(o_f64, np.float64)
    assert g.shape == o.shape, "%s: shape %s vs %s" % (what, g.shape, o.shape)
    err = np.abs(g - o)
    tol = CENTROID_RTOL * np.maximum(np.abs(o), 1e-2)
    if not (err <= tol).all():
        i = np.argmax(err - tol)
        raise AssertionError("%s: centroid off by %g (tol %g) at flat index %d" % (what, err.flat[i], tol.flat[i], i))
    return float((err / np.maximum(np.abs(o), 1e-2)).max()) if err.size else 0.0


# float32 unit roundoff: the bound of the error of one rounded float operation, relative to its exact result; and the
# absolute error of a result rounded in the subnormal range (half the spacing 2^-149), where the relative bound fails
U32 = 2.0 ** -24
ETA32 = 2.0 ** -150


def centroid_error_bound(xyzi, point_idx, voxel_idx, count):
    """Per voxel and component, the standard bound of a float32 centroid: the sum of n values in a fixed order is off by at
    most gamma_{n} * sum|x_i| (gamma_n = n u / (1 - n u)), and the division adds u * |centroid|. Returns
    (gamma_n * mean|x_i|) as an array [voxels, 4]; add U32 * |c| for the division."""
    x = np.abs(np.asarray(xyzi, np.float64))
    pidx = np.asarray(point_idx, np.int64)
    ok = pidx >= 0
    where = np.searchsorted(voxel_idx, pidx[ok])
    where = np.minimum(where, max(len(voxel_idx) - 1, 0))
    hit = np.asarray(voxel_idx, np.int64)[where] == pidx[ok]
    abs_sum = np.zeros((len(voxel_idx), 4))
    np.add.at(abs_sum, where[hit], x[ok][hit])
    n = np.asarray(count, np.float64)[:, None]
    gamma = n * U32 / (1.0 - n * U32)
    return gamma * abs_sum / n


def assert_centroids_within_bound(g, o_f64, xyzi, point_idx, voxel_idx, count, what=""):
    """|c_gpu - c_f64| <= gamma_n * mean|x_i| + u * |c_f64| (+ eta for a centroid that rounds to a subnormal) per component
    (centroid_error_bound): meaningful at any offset from the origin, unlike a relative tolerance, which at kilometres is
    wider than a voxel. Sums of subnormals are exact; only the division can round in the subnormal range."""
    g = np.asarray(g, np.float64)
    o = np.asarray(o_f64, np.float64)
    assert g.shape == o.shape, "%s: shape %s vs %s" % (what, g.shape, o.shape)
    if not g.size:
        return 0.0
    tol = centroid_error_bound(xyzi, point_idx, voxel_idx, count) + U32 * np.abs(o) + ETA32
    err = np.abs(g - o)
    if not (err <= tol).all():
        i = np.argmax(err - tol)
        raise AssertionError("%s: centroid off by %g (bound %g) at flat index %d" % (what, err.flat[i], tol.flat[i], i))
    return float((err / np.maximum(tol, 1e-300)).max())


def upload_segments(cm, frames, layout_of):
    """frames: list (per frame) of list (per sensor) of (xyzi, is_dense). Returns (segments, oracle cloud dicts per frame)."""
    items, per_frame = [], []
    for f, sensors in enumerate(frames):
        cds = []
        for s, (xyzi, dense) in enumerate(sensors):
            lt = layout_of(f, s)
            data = synth.pack_cloud(xyzi, *lt)
            buf = cm.upload(data if len(data) else np.zeros(16, np.uint8))
            items.append((buf.ptr, len(xyzi), make_layout(lt[0], lt[1], lt[2], lt[3], lt[4], dense), s, f))
            cds.append(dict(data=data, n_points=len(xyzi), point_step=lt[0], off_x=lt[1], off_y=lt[2], off_z=lt[3],
                            off_i=lt[4], is_dense=int(dense), m=cm.get_extrinsic(s)))
        per_frame.append(cds)
    return cm.make_segments(items), per_frame


def check_survivors(out, frames_info, oracle_frames):
    for f, (fi, o) in enumerate(zip(frames_info, oracle_frames)):
        sx = out["survivor_xyzi"][fi.survivor_begin:fi.survivor_end]
        ss = out["survivor_src"][fi.survivor_begin:fi.survivor_end]
        assert len(ss) == o["n_survivors"], "frame %d: %d survivors vs oracle %d" % (f, len(ss), o["n_survivors"])
        assert (ss == o["survivor_src"]).all(), "frame %d: surviving-point indices differ" % f
        assert_bit_equal(sx, o["survivor_xyzi"], "frame %d survivor coordinates" % f)


def check_voxels(out, frames_info, oracle_frames, check_membership=True):
    worst = 0.0
    idx_bits = out["key_idx_bits"]
    mask = (1 << idx_bits) - 1 if idx_bits < 64 else (1 << 64) - 1
    for f, (fi, o) in enumerate(zip(frames_info, oracle_frames)):
        v0, v1 = fi.voxel_begin, fi.voxel_end
        assert v1 - v0 == o["n_voxels"], "frame %d: %d voxels vs oracle %d" % (f, v1 - v0, o["n_voxels"])
        if o["n_survivors"]:
            assert list(fi.min_b) == o["min_b"].tolist() and list(fi.div_b) == o["div_b"].tolist(), "frame %d grid" % f
            assert fi.pcl_overflow == o["pcl_overflow"]
        assert (out["voxel_idx"][v0:v1].astype(np.int64) == o["idx"]).all(), "frame %d: voxel ids / order differ" % f
        assert (out["voxel_count"][v0:v1] == o["count"]).all(), "frame %d: voxel counts differ" % f
        assert_bit_equal(out["voxel_xyzi"][v0:v1], o["centroid"], "frame %d centroid vs float oracle (asc. index)" % f)
        worst = max(worst, assert_centroids_close(out["voxel_xyzi"][v0:v1], o["centroid_f64"], "frame %d centroid" % f))
        if check_membership:
            s0, s1 = fi.survivor_begin, fi.survivor_end
            keys = out["sorted_key"][s0:s1]
            pts = out["sorted_point"][s0:s1].astype(np.int64)
            assert (np.diff(keys.astype(np.float64)) >= 0).all() and (keys[1:] >= keys[:-1]).all(), "keys not sorted"
            assert ((keys >> np.uint64(idx_bits)) == f).all() if idx_bits < 64 else True
            member = np.full(s1 - s0, -2, np.int64)
            member[pts - s0] = (keys & np.uint64(mask)).astype(np.int64)
            assert (member == o["point_idx"]).all(), "frame %d: voxel membership differs" % f
            # stable sort: inside a voxel the points are in ascending index order
            same = keys[1:] == keys[:-1]
            assert (pts[1:][same] > pts[:-1][same]).all(), "sort is not stable"
    return worst


def reference_front_zones():
    """The ten PassThrough chains proceedFront runs on one ROI-cropped cloud (pc_preprocessing_main.cpp:228-270 with
    pcl_preprocessing/src/Parameter.h:31-55): five x windows [deviation, deviation + length] (float arithmetic), each
    followed by the ground window z in [-zg, zg] and the no-ground window z in [zg + 0.01, roi_z_max] -- the `+ 0.01` is
    a double addition narrowed to float by setFilterLimits (removeGround, :80-92)."""
    f32 = np.float32
    roi_mid, roi_z_max = f32(15), f32(3.0)
    front, mid, mid2, veh, rear = f32(30.0), f32(15.0), f32(11.0), f32(8.0), f32(11)
    parts = [  # (length, deviation, z_max_ground)
        (front, -roi_mid + rear + veh + mid + mid2, f32(2.5)),
        (mid2, -roi_mid + rear + veh + mid, f32(2.0)),
        (mid, -roi_mid + rear + veh, f32(1.5)),
        (veh, -roi_mid + rear, f32(0.3)),
        (rear, -roi_mid, f32(0.5)),
    ]
    zones = []
    for length, dev, zg in parts:
        x_pass = (0, float(f32(dev)), float(f32(dev) + f32(length)), 0)
        zones.append([x_pass, (2, float(-zg), float(zg), 0)])
        zones.append([x_pass, (2, float(f32(np.float64(zg) + 0.01)), float(roi_z_max), 0)])
    return zones
