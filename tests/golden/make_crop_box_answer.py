"""Writes tests/golden/crop_box.json: known answers of pcl::CropBox (PCL 1.8.1 CropBox::applyFilter) worked out point by
point with scalar float32 arithmetic written out here step by step -- no oracle code is imported. Coordinates are stored
as the hex bits of their float32 values, so -0.0, +-inf and NaN survive the trip.

Cases:
  ego_negative      a negative axis-aligned ego box, points exactly on each of the six faces and one ulp either side;
  yaw_rotated       a yawed + translated box (positive), points on and one ulp off its faces in the box frame;
  tiny_rotation     a 1e-6 rad yaw: the inverse is the identity within Eigen's 1e-5, so PCL skips the rotation
                    (a point one ulp outside stays outside; applying the rotation would move it inside);
  nan_dense / nan_nondense / nan_negative
                    NaN, +-inf and -0.0 rows with no PassThrough in front: a dense input keeps NaN rows in a positive box
                    (NaN is "inside"), a non-dense input drops every non-finite row, a negative box drops NaN rows.

Run: python tests/golden/make_crop_box_answer.py
"""
import ctypes
import ctypes.util
import json
import os

import numpy as np

F = np.float32
HERE = os.path.dirname(os.path.abspath(__file__))
_m = ctypes.CDLL(ctypes.util.find_library("m") or "libm.so.6")
_m.cosf.restype = _m.sinf.restype = ctypes.c_float
_m.cosf.argtypes = _m.sinf.argtypes = [ctypes.c_float]


def cosf(v):
    return F(_m.cosf(float(F(v))))


def sinf(v):
    return F(_m.sinf(float(F(v))))


def up(v, k=1):
    for _ in range(k):
        v = np.nextafter(F(v), F(np.inf))
    return F(v)


def down(v, k=1):
    for _ in range(k):
        v = np.nextafter(F(v), F(-np.inf))
    return F(v)


def hexf(v):
    return "%08x" % int(np.asarray(v, F).view(np.uint32))


def fuzzy_identity(rows):
    """Eigen isIdentity(1e-5): |d - 1| <= min(|d|, 1) * 1e-5 on the diagonal, |v| <= 1e-5 elsewhere."""
    for r in range(3):
        for c in range(4):
            v = F(rows[r][c])
            if r == c:
                if not abs(F(v - F(1))) <= F(min(abs(v), F(1)) * F(1e-5)):
                    return False
            elif not abs(v) <= F(1e-5):
                return False
    return True


def inverse_rotation(roll, pitch, yaw):
    a, b, c, d, e, f = cosf(yaw), sinf(yaw), cosf(pitch), sinf(pitch), cosf(roll), sinf(roll)
    de, df = F(d * e), F(d * f)
    m = [[F(a * c), F(F(a * df) - F(b * e)), F(F(b * f) + F(a * de))],
         [F(b * c), F(F(a * e) + F(b * df)), F(F(b * de) - F(a * f))],
         [F(-d), F(c * f), F(c * e)]]

    def cof(i, j):
        i1, i2, j1, j2 = (i + 1) % 3, (i + 2) % 3, (j + 1) % 3, (j + 2) % 3
        return F(F(m[i1][j1] * m[i2][j2]) - F(m[i1][j2] * m[i2][j1]))
    det = F(F(F(cof(0, 0) * m[0][0]) + F(cof(1, 0) * m[1][0])) + F(cof(2, 0) * m[2][0]))
    invdet = F(F(1) / det)
    inv = [[F(cof(j, i) * invdet) for j in range(3)] for i in range(3)]
    for i in range(3):
        # -(linear) * (0, 0, 0): a signed zero
        inv[i].append(F(F(F(-inv[i][0]) * F(0)) + F(F(-inv[i][1]) * F(0))) + F(F(-inv[i][2]) * F(0)))
    return inv


def row(m, r, x, y, z):
    return F(F(F(F(m[r][0] * x) + F(m[r][1] * y)) + F(m[r][2] * z)) + m[r][3])


def kept(points, is_dense, box):
    mn, mx = [F(v) for v in box["min"]], [F(v) for v in box["max"]]
    t = [[F(v) for v in box["transform"][4 * r:4 * r + 4]] for r in range(3)]
    tr = [F(v) for v in box["translation"]]
    rot = [F(v) for v in box["rotation"]]
    use_t = not fuzzy_identity(t)
    use_tr = any(v != 0 for v in tr)
    inv = inverse_rotation(*rot) if any(v != 0 for v in rot) else None
    use_r = inv is not None and not fuzzy_identity(inv)
    out = []
    with np.errstate(all="ignore"):
        for i, (x, y, z) in enumerate(points):
            x, y, z = F(x), F(y), F(z)
            if not is_dense and not (np.isfinite(x) and np.isfinite(y) and np.isfinite(z)):
                continue
            if use_t:
                x, y, z = row(t, 0, x, y, z), row(t, 1, x, y, z), row(t, 2, x, y, z)
            if use_tr:
                x, y, z = F(x - tr[0]), F(y - tr[1]), F(z - tr[2])
            if use_r:
                x, y, z = row(inv, 0, x, y, z), row(inv, 1, x, y, z), row(inv, 2, x, y, z)
            outside = x < mn[0] or y < mn[1] or z < mn[2] or x > mx[0] or y > mx[1] or z > mx[2]
            if outside == bool(box["negative"]):
                out.append(i)
    return out


IDENT = [1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0]


def box(mn, mx, translation=(0.0, 0.0, 0.0), rotation=(0.0, 0.0, 0.0), transform=IDENT, negative=False):
    return dict(min=[float(F(v)) for v in mn], max=[float(F(v)) for v in mx], translation=[float(F(v)) for v in translation],
                rotation=[float(F(v)) for v in rotation], transform=[float(F(v)) for v in transform], negative=int(negative))


def face_points(mn, mx, centre):
    """Points exactly on each face of [mn, mx] and one ulp either side of it, the other coordinates at the centre."""
    pts = []
    for a in range(3):
        for face in (mn[a], mx[a]):
            for v in (down(face), F(face), up(face)):
                p = [F(c) for c in centre]
                p[a] = v
                pts.append(p)
    return pts


def main():
    cases = []
    # ego box of a car (x forward): removed by a negative box; faces hit exactly and one ulp off
    mn, mx = (F(-1.25), F(-1.0), F(-0.5)), (F(3.75), F(1.0), F(1.75))
    pts = face_points(mn, mx, (F(1.0), F(0.0), F(0.5))) + [[F(10), F(0), F(0)], [F(0), F(5), F(0)], [F(0), F(0), F(3)],
                                                             [F(-0.0), F(-0.0), F(-0.0)]]
    cases.append(dict(name="ego_negative", is_dense=1, box=box(mn, mx, negative=True), points=pts))
    # yawed + translated box: the box frame of a point is R^-1 (p - t); put points on its faces in that frame by walking
    # world x one ulp at a time until the local coordinate lands on the face, then one ulp either side
    bx = box((-1.0, -0.5, -1.0), (1.0, 0.5, 1.0), translation=(2.0, 1.0, 0.0), rotation=(0.0, 0.0, 0.5))
    inv = inverse_rotation(*[F(v) for v in bx["rotation"]])
    tr = [F(v) for v in bx["translation"]]
    pts = []
    c5, s5 = float(np.cos(0.5)), float(np.sin(0.5))
    for a in range(3):
        for face in (bx["min"][a], bx["max"][a]):
            loc = [0.0, 0.0, 0.0]
            loc[a] = face
            w = [c5 * loc[0] - s5 * loc[1] + 2.0, s5 * loc[0] + c5 * loc[1] + 1.0, loc[2]]
            x0 = F(w[0])
            for k in range(-64, 65):
                x = up(x0, k) if k >= 0 else down(x0, -k)
                p = [x, F(w[1]), F(w[2])]
                q = [F(p[0] - tr[0]), F(p[1] - tr[1]), F(p[2] - tr[2])]
                lv = row(inv, a, *q)
                if lv in (down(F(face)), F(face), up(F(face))):
                    pts.append(p)
    pts += [[F(2), F(1), F(0)], [F(0), F(0), F(0)], [F(2.5), F(1.2), F(0.9)]]
    cases.append(dict(name="yaw_rotated", is_dense=1, box=bx, points=pts))
    # 1e-6 rad of yaw: skipped by PCL. y one ulp above max at x = 100 stays outside (a rotation would move it ~1e-4 in)
    bt = box((-200.0, -1.0, -1.0), (200.0, 1.0, 1.0), rotation=(0.0, 0.0, 1e-6))
    cases.append(dict(name="tiny_rotation", is_dense=1, box=bt,
                      points=[[F(100), up(F(1)), F(0)], [F(100), F(1), F(0)], [F(-100), down(F(-1)), F(0)], [F(0), F(0), F(0)]]))
    nan, inf = F(np.nan), F(np.inf)
    rows = [[F(0.5), F(0.5), F(0.5)], [nan, F(0), F(0)], [F(0), nan, F(0)], [F(0), F(0), inf], [-inf, F(0), F(0)],
            [F(-0.0), F(0.0), F(-0.0)], [F(5), F(5), F(5)], [F(0), F(0), nan]]
    pos = box((-1.0, -1.0, -1.0), (1.0, 1.0, 1.0))
    cases.append(dict(name="nan_dense", is_dense=1, box=pos, points=rows))
    cases.append(dict(name="nan_nondense", is_dense=0, box=pos, points=rows))
    cases.append(dict(name="nan_negative", is_dense=1, box=box((-1.0, -1.0, -1.0), (1.0, 1.0, 1.0), negative=True), points=rows))
    out = []
    for c in cases:
        out.append(dict(name=c["name"], is_dense=c["is_dense"], box=c["box"],
                        points=[[hexf(v) for v in p] for p in c["points"]], kept=kept(c["points"], c["is_dense"], c["box"])))
    with open(os.path.join(HERE, "crop_box.json"), "w") as f:
        json.dump({"source": "tests/golden/make_crop_box_answer.py", "cases": out}, f, indent=1)
        f.write("\n")
    for c in out:
        print(c["name"], len(c["points"]), "points, kept", c["kept"])


if __name__ == "__main__":
    main()
