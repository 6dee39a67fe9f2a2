"""CPU tests of the pcl::CropBox statements (not gpu): the C++ oracle (tests/crop_box_oracle.cpp), the numpy restatement
(tests/crop_box_np.py) and the known answers of tests/golden/crop_box.json (worked out step by step) agree bit for bit;
Eigen's fuzzy identity decides whether a step runs; the C-ABI struct and its ctypes mirrors have one layout."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import crop_box_cases as K
import crop_box_np
from crop_box_oracle import crop_box

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("case", [c["name"] for c in K.golden()])
def test_golden_known_answers(case):
    c = next(c for c in K.golden() if c["name"] == case)
    want = np.asarray(c["kept"], np.int64)
    got_cpp = crop_box(c["xyzi"], bool(c["is_dense"]), c["box"])
    got_np = np.nonzero(crop_box_np.crop_box_mask(c["xyzi"], bool(c["is_dense"]), c["box"]))[0]
    assert np.array_equal(got_cpp, want), (case, got_cpp, want)
    assert np.array_equal(got_np, want), (case, got_np, want)


@pytest.mark.parametrize("name", sorted(K.BOXES))
@pytest.mark.parametrize("is_dense", [1, 0])
def test_oracle_and_numpy_agree_on_edge_clouds(name, is_dense):
    b = K.BOXES[name]
    x = K.edge_cloud(7 + len(name), b)
    hits = K.face_hits(x, b)
    assert all(h > 0 for h in hits), "every face gets exact hits: %s" % hits
    got_cpp = crop_box(x, bool(is_dense), b)
    got_np = np.nonzero(crop_box_np.crop_box_mask(x, bool(is_dense), b))[0]
    assert np.array_equal(got_cpp, got_np)
    nonfinite = ~np.isfinite(x[:, :3]).all(1)
    kept_nf = np.isin(np.nonzero(nonfinite)[0], got_cpp)
    if not is_dense:
        assert not kept_nf.any(), "a non-dense input loses every non-finite point"
    else:
        nan_rows = np.isnan(x[:, :3]).any(1)
        assert np.isin(np.nonzero(nan_rows)[0], got_cpp).all() != b["negative"], "NaN counts as inside"


@pytest.mark.parametrize("side", ["below", "above"])
def test_fuzzy_identity_decides_the_steps(side):
    """Eigen's isIdentity(1e-5): off the diagonal |v| <= 1e-5, on it |d - 1| <= min(|d|, 1) * 1e-5. A step whose matrix
    passes is skipped, so a point one ulp outside a face stays outside; one that fails is applied and moves the point."""
    eps = np.float32(0.99e-5) if side == "below" else np.float32(1.01e-5)
    skip = side == "below"
    # off-diagonal entry of setTransform: y' = eps * x + y; at x = 1000 that moves y by about 1e-2
    t = np.eye(3, 4, dtype=np.float32)
    t[1, 0] = eps
    assert crop_box_np.is_identity(t) == skip
    b = K.box((-2000.0, -1.0, -1.0), (2000.0, 1.0, 1.0), transform=t)
    # inside as given and outside once the step is applied; the other point is outside either way
    pts = np.array([[1000.0, 0.995, 0.0, 0.0], [1000.0, np.nextafter(np.float32(1), np.float32(2)), 0.0, 0.0]], np.float32)
    got = crop_box(pts, True, b)
    assert np.array_equal(got, np.nonzero(crop_box_np.crop_box_mask(pts, True, b))[0])
    assert got.tolist() == ([0] if skip else [])
    # diagonal entry: relative compare
    t2 = np.eye(3, 4, dtype=np.float32)
    t2[0, 0] = np.float32(1) + eps
    assert crop_box_np.is_identity(t2) == skip
    b2 = K.box((-1.0, -1.0, -1.0), (1000.0, 1.0, 1.0), transform=t2)
    p2 = np.array([[1000.0, 0.0, 0.0, 0.0]], np.float32)
    assert crop_box(p2, True, b2).tolist() == ([0] if skip else [])
    # the rotation: a yaw of eps rad gives an inverse with off-diagonal -+sin(eps)
    inv = crop_box_np.rotation_inverse(0.0, 0.0, eps)
    assert crop_box_np.is_identity(inv) == (abs(inv[0, 1]) <= np.float32(1e-5))
    b3 = K.box((-2000.0, -1.0, -1.0), (2000.0, 1.0, 1.0), rotation=(0.0, 0.0, float(eps)))
    p3 = np.array([[-1000.0, 0.995, 0.0, 0.0]], np.float32)   # y_local = -sin * x + cos * y: pushed out when applied
    assert crop_box(p3, True, b3).tolist() == ([0] if crop_box_np.is_identity(inv) else [])
    assert np.array_equal(crop_box(p3, True, b3), np.nonzero(crop_box_np.crop_box_mask(p3, True, b3))[0])


def test_steps_are_not_composed():
    """transform, translation and rotation run one after another: on the edge clouds of a box that uses all three, the
    single composed matrix keeps a different set of points (so a composed implementation would be caught)."""
    b = K.BOXES["transform_neg"]
    b = dict(b, translation=(0.375, -0.625, 0.25), rotation=(0.2, 0.05, -0.4))
    x = K.edge_cloud(99, b, special=False)
    seq = crop_box(x, True, b)
    inv = crop_box_np.rotation_inverse(*b["rotation"]).astype(np.float64)
    t = np.asarray(b["transform"], np.float64)
    tr = np.asarray(b["translation"], np.float64)
    A = inv[:, :3] @ t[:, :3]
    c = inv[:, :3] @ (t[:, 3] - tr) + inv[:, 3]
    m = np.concatenate([A, c[:, None]], 1).astype(np.float32)
    with np.errstate(all="ignore"):
        loc = np.stack([((m[r, 0] * x[:, 0] + m[r, 1] * x[:, 1]) + m[r, 2] * x[:, 2]) + m[r, 3] for r in range(3)], 1)
    mn, mx = np.asarray(b["min"], np.float32), np.asarray(b["max"], np.float32)
    outside = ((loc < mn) | (loc > mx)).any(1)
    composed = np.nonzero(outside)[0]
    assert not np.array_equal(seq, composed)


def test_crop_box_struct_layout():
    """cm_crop_box_t (include/cloud_merger_gpu.h), the library's ctypes mirror and the oracle's cmo_crop_box_t agree."""
    from cloud_merger_b200 import _lib
    import crop_box_oracle
    src = r'''
#include <stddef.h>
#include <stdio.h>
#include "cloud_merger_gpu.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %d\n", sizeof(cm_crop_box_t), offsetof(cm_crop_box_t, max), offsetof(cm_crop_box_t, translation),
         offsetof(cm_crop_box_t, rotation), offsetof(cm_crop_box_t, transform), offsetof(cm_crop_box_t, negative),
         offsetof(cm_crop_box_t, reserved), CM_MAX_CROP_BOXES);
  return 0;
}'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(v) for v in subprocess.check_output([exe]).split()]
    for T in (_lib.CmCropBox, crop_box_oracle.CmoCropBox):
        want = [C.sizeof(T)] + [getattr(T, f).offset for f in ("max", "translation", "rotation", "transform", "negative",
                                                               "reserved")] + [_lib.CM_MAX_CROP_BOXES]
        assert got == want, (T.__name__, got, want)
