"""Inputs and expectations of the pcl::CropBox tests (tests only): the boxes, edge clouds with points on every face and a few
ulps either side of it in the box frame, and the merged-frame expectation transform -> passes -> boxes -> concat ->
VoxelGrid composed from the float oracle's stages (oracle/cm_oracle.cpp, tests/crop_box_oracle.cpp)."""
from __future__ import annotations

import json
import os

import numpy as np

import crop_box_np
import crop_box_oracle

F32 = np.float32
HERE = os.path.dirname(os.path.abspath(__file__))
IDENT = np.eye(3, 4, dtype=F32)


def box(mn, mx, translation=(0.0, 0.0, 0.0), rotation=(0.0, 0.0, 0.0), transform=None, negative=False) -> dict:
    return dict(min=tuple(float(F32(v)) for v in mn), max=tuple(float(F32(v)) for v in mx),
                translation=tuple(float(F32(v)) for v in translation), rotation=tuple(float(F32(v)) for v in rotation),
                transform=(IDENT if transform is None else np.asarray(transform, F32).reshape(3, 4)).copy(),
                negative=bool(negative))


def to_cm(b: dict):
    """The library's cm_crop_box_t of a box dict."""
    from cloud_merger_b200 import make_crop_box
    return make_crop_box(b["min"], b["max"], b["translation"], b["rotation"], b["transform"], b["negative"])


def _tilt():
    t = np.eye(3, 4, dtype=F32)
    c, s = F32(np.cos(0.3)), F32(np.sin(0.3))
    t[0, 0], t[0, 2], t[2, 0], t[2, 2] = c, s, -s, c
    t[:, 3] = (F32(0.25), F32(-0.5), F32(0.125))
    return t


# an ego box (negative, translated + yawed like a car parked at an angle to the base frame), a roof rack, a mirror, ...
EGO = box((-2.25, -1.0, -0.75), (2.5, 1.0, 1.5), translation=(1.25, 0.0, 0.5), rotation=(0.0, 0.0, 0.15), negative=True)
BOXES = {
    "ego": EGO,
    "axis_pos": box((-4.0, -3.0, -1.0), (6.0, 3.0, 2.0)),
    "axis_neg": box((-1.5, -1.0, -0.5), (3.5, 1.0, 1.25), negative=True),
    "rpy_pos": box((-2.0, -1.5, -0.75), (2.0, 1.5, 0.75), translation=(0.5, -0.25, 0.0), rotation=(0.1, -0.2, 0.7)),
    "transform_neg": box((-1.0, -1.0, -1.0), (1.5, 1.0, 1.0), transform=_tilt(), rotation=(0.0, 0.05, 0.0), negative=True),
    "tiny_rot_pos": box((-5.0, -2.0, -2.0), (5.0, 2.0, 2.0), rotation=(0.0, 0.0, 1e-6)),
}


def local_of(xyz, b):
    """The box-frame coordinates the numpy CropBox compares (steps 2-4)."""
    x, y, z = (np.asarray(xyz[:, k], F32) for k in range(3))
    with np.errstate(all="ignore"):
        def apply(m, x, y, z):
            return tuple(((m[r, 0] * x + m[r, 1] * y) + m[r, 2] * z) + m[r, 3] for r in range(3))
        if not crop_box_np.is_identity(b["transform"]):
            x, y, z = apply(np.asarray(b["transform"], F32), x, y, z)
        tr = np.asarray(b["translation"], F32)
        if (tr != 0).any():
            x, y, z = x - tr[0], y - tr[1], z - tr[2]
        if (np.asarray(b["rotation"], F32) != 0).any():
            inv = crop_box_np.rotation_inverse(*b["rotation"])
            if not crop_box_np.is_identity(inv):
                x, y, z = apply(inv, x, y, z)
    return np.stack([x, y, z], 1)


def _world_of(loc, b):
    """float64 inverse of steps 2-4 (a guess the ulp walk then corrects)."""
    r, p, yw = (float(v) for v in b["rotation"])
    cr, sr, cp, sp, cy, sy = np.cos(r), np.sin(r), np.cos(p), np.sin(p), np.cos(yw), np.sin(yw)
    R = np.array([[cy * cp, cy * sp * sr - sy * cr, sy * sr + cy * sp * cr],
                  [sy * cp, cy * cr + sy * sp * sr, sy * sp * cr - cy * sr],
                  [-sp, cp * sr, cp * cr]])
    w = loc.astype(np.float64) @ R.T + np.asarray(b["translation"], np.float64)
    t = np.asarray(b["transform"], np.float64)
    if not crop_box_np.is_identity(b["transform"]):
        w = (w - t[:, 3]) @ np.linalg.inv(t[:, :3]).T
    return w


def edge_cloud(seed: int, b: dict, n_face: int = 24, n_random: int = 3000, special: bool = True) -> np.ndarray:
    """xyzi points on every face of b and 1-3 ulps either side of it in the box frame, plus random points around the box,
    plus (special) -0.0, +-inf and NaN rows. World coordinates are walked one ulp at a time until the box-frame coordinate
    is exactly on the face or within 3 ulps of it."""
    rng = np.random.default_rng(seed)
    mn, mx = np.asarray(b["min"], F32), np.asarray(b["max"], F32)
    out = []
    for a in range(3):
        for face in (mn[a], mx[a]):
            loc = rng.uniform(mn, mx, size=(n_face, 3))
            loc[:, a] = face
            w = _world_of(loc, b).astype(F32)
            cand = [w]
            for ax in range(3):
                for k in range(1, 48):
                    for sgn in (1, -1):
                        c = w.copy()
                        c[:, ax] = c[:, ax] + sgn * k * np.spacing(np.abs(c[:, ax])).astype(F32)
                        cand.append(c)
            cand = np.concatenate(cand)
            lv = local_of(cand, b)[:, a]
            dist = np.abs(lv.view(np.int32).astype(np.int64) - F32(face).view(np.int32).astype(np.int64))
            same_sign = np.signbit(lv) == np.signbit(F32(face))
            out.append(cand[(dist <= 3) & same_sign])
    pts = np.concatenate(out)
    rng.shuffle(pts)
    centre = (mn + mx) / 2
    span = (mx - mn) * 1.5 + 1.0
    rnd = _world_of(rng.uniform(centre - span, centre + span, size=(n_random, 3)).astype(F32), b).astype(F32)
    xyz = np.concatenate([pts, rnd])
    x = np.zeros((len(xyz), 4), F32)
    x[:, :3] = xyz
    x[:, 3] = rng.uniform(0, 255, len(x)).astype(F32)
    if special:
        sp = np.array([[-0.0, -0.0, -0.0, 1], [0.0, -0.0, 0.0, 2], [np.nan, 0, 0, 3], [0, np.nan, 0, 4], [0, 0, np.nan, 5],
                       [np.inf, 0, 0, 6], [0, -np.inf, 0, 7], [0, 0, np.inf, 8], [np.nan, np.nan, np.nan, 9]], F32)
        x = np.concatenate([x, sp])
        rng.shuffle(x)
    return x


def face_hits(x, b):
    """Number of points exactly on each of the six faces (box frame)."""
    loc = local_of(x[:, :3], b)
    mn, mx = np.asarray(b["min"], F32), np.asarray(b["max"], F32)
    return [int((loc[:, a] == f).sum()) for a in range(3) for f in (mn[a], mx[a])]


def golden():
    with open(os.path.join(HERE, "golden", "crop_box.json")) as f:
        d = json.load(f)
    for c in d["cases"]:
        pts = np.array([[int(h, 16) for h in p] for p in c["points"]], np.uint32).view(F32)
        x = np.zeros((len(pts), 4), F32)
        x[:, :3] = pts
        c["xyzi"] = x
        b = c["box"]
        c["box"] = box(b["min"], b["max"], b["translation"], b["rotation"], np.asarray(b["transform"], F32).reshape(3, 4),
                       bool(b["negative"]))
    return d["cases"]


def merge_expectation(oracle, clouds, passes, boxes, leaf, min_points=1, downsample_all=True, force64=True):
    """The float oracle's merged frame with CropBox stages: per sensor unpack -> transform -> PassThrough chain (each
    stage copies its survivors) -> boxes in order (the first box sees the sensor's is_dense when no pass ran, every later
    stage a dense cloud) -> concat in sensor order -> VoxelGrid. Non-finite survivors (a dense cloud without passes, or a
    negative box that keeps +-inf) are skipped by the VoxelGrid, as the library does."""
    sx, ss, base = [], [], 0
    for c in clouds:
        p = oracle.unpack(c["data"], c["n_points"], c["point_step"], c["off_x"], c["off_y"], c["off_z"], c["off_i"])
        t = oracle.transform(p, c["m"], bool(c["is_dense"]))
        idx = np.arange(len(t), dtype=np.int64)
        cur = t
        for (axis, lo, hi, neg) in passes:
            k = oracle.passthrough(cur, int(axis), float(F32(lo)), float(F32(hi)), bool(neg)).astype(np.int64)
            cur, idx = np.ascontiguousarray(cur[k]), idx[k]
        dense = bool(c["is_dense"]) or len(passes) > 0
        for b in boxes:
            k = crop_box_oracle.crop_box(cur, dense, b).astype(np.int64)
            cur, idx = np.ascontiguousarray(cur[k]), idx[k]
            dense = True
        sx.append(cur)
        ss.append(base + idx)
        base += c["n_points"]
    sx = np.concatenate(sx) if sx else np.zeros((0, 4), F32)
    ss = np.concatenate(ss).astype(np.uint32)
    fin = np.isfinite(sx[:, :3]).all(1)
    v = oracle.voxelgrid(sx, [leaf] * 3, min_points, downsample_all, force64=force64, is_dense=bool(fin.all()))
    v.update(survivor_xyzi=sx, survivor_src=ss, n_survivors=len(sx), n_voxels=v["n"])
    return v
