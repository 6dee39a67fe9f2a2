"""CPU tests of the normal estimation's statements (no GPU): the C++ statement of PCL's loop (tests/ne_oracle.cpp) against
the numpy/scipy statement and the hand-worked golden answers, the branches of pcl::eigen33 each case family was built for,
the order of ties, and the trig rule of cm_ne_math.h against correctly rounded references and the host libm."""
import json
import os

import numpy as np
import pytest

import ne_cases as K
import ne_np as NP
import ne_oracle as O

F32 = np.float32
HERE = os.path.dirname(os.path.abspath(__file__))


def bits(a):
    return np.ascontiguousarray(a, F32).view(np.uint32)


@pytest.mark.parametrize("name,make,radius,vp", [
    ("eigen", lambda: K.eigen_family(1, 0.3), 0.3, (0.5, -0.5, 2.0)),
    ("small", lambda: K.small_groups(0.3), 0.3, (0.0, 0.0, 0.0)),
    ("lattice", lambda: K.lattice(8, 0.25), 0.3, (1.0, 1.0, 1.0)),
    ("ulp", lambda: K.ulp_edges(3, 0.1), 0.1, (0.0, 0.0, 5.0)),
    ("dups", lambda: K.with_duplicates(K.with_nonfinite(K.blobs(4, 1500), 4), 4, 0.3), 0.4, (0.0, 0.0, 0.0)),
    ("faces", lambda: K.shell_faces(11, float(F32(0.25) * F32(1.00390625))), 0.25, (0.0, 0.0, 0.0)),
])
def test_statements_agree_bit_for_bit(name, make, radius, vp):
    c = make()
    NP.check_slack(c, radius, NP.neighbour_lists(c, radius))
    grid = O.normals(c, radius, vp)
    assert (bits(grid) == bits(O.normals(c, radius, vp, exhaustive=True))).all(), "grid vs exhaustive"
    assert (bits(grid) == bits(NP.normals(c, radius, vp))).all(), "C++ vs numpy"


def test_roi_statements_agree():
    c = K.roi_cloud(7, 32, 1024)
    for r in (0.1, 0.3):
        NP.check_slack(c, r, NP.neighbour_lists(c, r))
        assert (bits(O.normals(c, r, (0.0, 0.0, 1.8))) == bits(NP.normals(c, r, (0.0, 0.0, 1.8)))).all(), r


def test_every_eigen33_branch_is_reached():
    _, cnt, paths, _ = O.normals(K.eigen_family(1, 0.3), 0.3, details=True)
    for b in (O.ROOTS2, O.TRIG, O.Q_CLAMP, O.ROOT0_NEG, O.PICK1, O.PICK2, O.PICK3, O.FLIP):
        assert ((paths & b) != 0).any(), b
    _, _, lat_paths, _ = O.normals(K.lattice(8, 0.25), 0.3, details=True)
    assert ((lat_paths & O.Q_CLAMP) != 0).any()
    # exact planes take computeRoots2 through |c0| < eps: planar data alone never reaches the closed form
    plane = K.cloud(np.column_stack([np.random.default_rng(2).uniform(0, 1, (400, 2)), np.zeros(400)]))
    _, _, pp, _ = O.normals(plane, 0.2, details=True)
    assert (pp[pp != 0] & O.ROOTS2).all() and not (pp & O.TRIG).any()


def test_small_groups_and_degenerate_sets():
    c = K.small_groups(0.3)
    out, cnt, _, _ = O.normals(c, 0.3, details=True)
    few = cnt < 3
    assert few.any() and (bits(out[few]) == 0x7FC00000).all()
    dup = np.arange(len(c))[-3:]  # three duplicates: zero covariance, NaN normal, curvature 0
    assert (bits(out[dup, :3]) == 0x7FC00000).all() and (out[dup, 3] == 0).all()


def test_ties_follow_the_index_order():
    """a lattice point's six neighbours at one distance: summing them ordered by d2 alone (stable in the order of the
    candidates) or by any other index order changes the bits of some normals; FLANN's (d2, index) is the rule"""
    c = K.lattice(6, 0.25) + np.array([0.37, 1.1, -0.6, 0], F32)
    lists = NP.neighbour_lists(c, 0.3)
    want = NP.normals(c, 0.3)
    rng = np.random.default_rng(0)
    changed = 0
    for i in range(len(c)):
        order = lists[i]
        a = c[order, :3]
        d2 = ((a - c[i, :3]) ** 2).sum(1)
        alt = order[np.lexsort((rng.permutation(len(order)), d2.astype(F32)))]
        s = np.zeros(9, F32)
        for j in alt:
            x, y, z = c[j, :3]
            for k, v in enumerate((x * x, x * y, x * z, y * y, y * z, z * z, x, y, z)):
                s[k] = F32(s[k] + F32(v))
        o, _ = O.solve(s[None], [len(alt)], c[i:i + 1])
        changed += int((bits(o[0]) != bits(want[i])).any())
    assert changed > 0


def test_golden_answers():
    g = json.load(open(os.path.join(HERE, "golden", "ne.json")))
    for case in g["cases"]:
        pts = np.array(case["xyzi"], F32).reshape(-1, 4)
        got = O.normals(pts, case["radius"], case["viewpoint"])
        assert bits(got).tolist() == case["bits"], case["name"]


def _random_neighbourhoods(seed, n):
    """(sums, count, query) of n random noisy planar patches, in FLANN's order as the statement forms them"""
    rng = np.random.default_rng(seed)
    for _ in range(n):
        m = int(rng.integers(5, 40))
        xyz = (rng.normal(size=(m, 3)) * np.array([0.2, 0.15, 0.01]) @ np.linalg.qr(rng.normal(size=(3, 3)))[0]
               + rng.uniform(-20, 20, 3)).astype(F32)
        s = np.zeros(9, F32)
        for x, y, z in xyz:
            for k, v in enumerate((x * x, x * y, x * z, y * y, y * z, z * z, x, y, z)):
                s[k] = F32(s[k] + F32(v))
        yield s, m, xyz[0]


def test_squared_norm_order_through_solve():
    """Eigen 3.3 sums a 3-vector as a0 + (a1 + a2) (redux_novec_unroller); on neighbourhoods where (a0 + a1) + a2 gives
    other bits, the shared solve gives Eigen's"""
    found = 0
    for s, m, q in _random_neighbourhoods(1, 3000):
        eig = NP.solve(s, m, q, (0, 0, 0), norm_order="eigen")
        left = NP.solve(s, m, q, (0, 0, 0), norm_order="left")
        if bits(np.array(eig)).tolist() == bits(np.array(left)).tolist():
            continue
        got, _ = O.solve(s[None], [m], np.append(q, 0)[None])
        assert bits(got[0]).tolist() == bits(np.array(eig)).tolist()
        found += 1
    assert found >= 5


def test_flip_sums_left_to_right():
    """flipNormalTowardsViewpoint's float& overload sums (vx*nx + vy*ny) + vz*nz; viewpoints near the tangent plane where
    Eigen's a0 + (a1 + a2) would decide the flip the other way: the shared solve decides as PCL does"""
    rng = np.random.default_rng(3)
    found = 0
    for s, m, q in _random_neighbourhoods(2, 400):
        n = np.array(NP.solve(s, m, q, (0, 0, 0))[:3], F32)
        if not np.isfinite(n).all() or (np.abs(n) < 1e-3).any():
            continue
        for _ in range(60):
            t = F32(rng.uniform(0.5, 4.0))
            d = np.array([t / n[0], -t / n[1], F32(rng.uniform(-1, 1)) * F32(2.0 ** -rng.integers(18, 30)) / n[2]], F32)
            vp = (q + d).astype(F32)
            pcl = NP.solve(s, m, q, vp, flip_order="pcl")
            eig = NP.solve(s, m, q, vp, flip_order="eigen")
            if bits(np.array(pcl)).tolist() == bits(np.array(eig)).tolist():
                continue
            got, paths = O.solve(s[None], [m], np.append(q, 0)[None], vp)
            assert bits(got[0]).tolist() == bits(np.array(pcl)).tolist()
            found += 1
    assert found >= 5


def test_hand_derived_planes_and_tetrahedron():
    """Exact planes z = 0: xz, yz and zz vanish, so c0 = 0 and computeRoots2 gives roots[0] = 0; the third row of the
    shifted matrix is 0, so only row0 x row1 = (xy * 0 - 0 * yy, 0 * xy - xx * 0, xx * yy - xy * xy) is non-zero, and
    sqrt(fl(d^2)) = |d| makes it (+-0, +-0, 1) exactly: the zeros carry the sign of xy (fl(xy * 0) - (+0)). The
    eigenvalue is 0, so the curvature is 0. Flipping multiplies by -1, zeros included."""
    tri = K.cloud([[0, 0, 0], [0.1, 0, 0], [0, 0.1, 0]])        # cov xy = 0 - mx * my < 0: the zeros are -0
    up = O.normals(tri, 0.5, (0, 0, 1))
    assert bits(up).tolist() == [[0x80000000, 0x80000000, 0x3F800000, 0]] * 3
    down = O.normals(tri, 0.5, (0, 0, -1))
    assert bits(down).tolist() == [[0, 0, 0xBF800000, 0]] * 3
    pos = K.cloud([[0, 0, 0], [0.1, 0.1, 0], [0.2, 0.1, 0]])    # cov xy > 0: +0
    assert bits(O.normals(pos, 0.5, (0, 0, 1))).tolist() == [[0, 0, 0x3F800000, 0]] * 3
    # a tetrahedron: the closed form; against a double-precision eigen decomposition of the same covariance
    tet = np.array([[0, 0, 0], [0.1, 0, 0], [0, 0.1, 0], [0, 0, 0.05]])
    c = np.cov(tet.T, bias=True)
    w, v = np.linalg.eigh(c)
    got = O.normals(K.cloud(tet), 0.5, (1.0, 1.0, 1.0))
    for p, row in zip(tet, got):
        assert abs(abs(float(np.dot(row[:3], v[:, 0]))) - 1.0) < 1e-6
        assert float(row[:3] @ (np.array([1.0, 1.0, 1.0]) - p)) > 0  # turned towards the viewpoint
        assert abs(row[3] - w[0] / w.sum()) < 1e-6


# ---- the trig rule ------------------------------------------------------------------------------------------------------
def test_cos_sin_exhaustive_on_theta_range():
    """every float theta in [0, fl(fl(pi) * fl(1/3))]: the rule is the correctly rounded float; its agreement with this
    host's sinf / cosf is reported"""
    top = F32(F32(np.pi) * F32(1.0 / 3.0))
    st = O.sincos_check(0, int(np.array(top, F32).view(np.uint32)))
    print("\ntrig rule vs correctly rounded, %d floats: %r" % (st["floats"], st))
    print("host libm agrees: sinf %.4f %%, cosf %.4f %%" % (100.0 * st["sinf_same"] / st["floats"],
                                                            100.0 * st["cosf_same"] / st["floats"]))
    assert st["sin_bad"] == 0 and st["cos_bad"] == 0 and st["sign_bad"] == 0
    assert st["unresolved"] < 100
    assert st["sinf_same"] > 0.99 * st["floats"] and st["cosf_same"] > 0.99 * st["floats"]


def test_atan2_sampled():
    st = O.atan2_check(7, 10 ** 8)
    print("\natan2 rule vs correctly rounded: %r; atan2f agrees on %.2f %%" % (st, 100.0 * st["atan2f_same"] / st["samples"]))
    assert st["bad"] == 0 and st["unresolved"] < 100
    assert st["atan2f_same"] > 0.7 * st["samples"]


def test_atan2_special_values():
    inf, nan = float("inf"), float("nan")
    pi, pi2, pi4 = F32(np.pi), F32(np.pi / 2), F32(np.pi / 4)
    cases = [(0.0, 1.0, 0.0), (-0.0, 1.0, -0.0), (0.0, 0.0, 0.0), (-0.0, 0.0, -0.0), (0.0, -0.0, pi), (-0.0, -0.0, -pi),
             (0.0, -1.0, pi), (-0.0, -1.0, -pi), (1.0, 0.0, pi2), (-1.0, -0.0, -pi2), (inf, 1.0, pi2), (-inf, -1.0, -pi2),
             (inf, inf, pi4), (-inf, inf, -pi4), (inf, -inf, F32(3 * np.pi / 4)), (-inf, -inf, -F32(3 * np.pi / 4)),
             (1.0, inf, 0.0), (-1.0, inf, -0.0), (1.0, -inf, pi), (-1.0, -inf, -pi), (1.0, 1.0, pi4),
             (1e-45, 1e38, 0.0), (1e38, 1e-45, pi2)]
    for y, x, w in cases:
        got = O.atan2(y, x)
        assert bits(np.array([got])) == bits(np.array([w], F32)), (y, x, got, w)
    for y, x in ((nan, 1.0), (1.0, nan), (nan, nan)):
        assert bits(np.array([O.atan2(y, x)]))[0] == 0x7FC00000
    for x in (0.0, -0.0, 1e-30, -1e-30, 0.5, -1.04):
        assert bits(np.array([O.sin(-x)]))[0] == bits(np.array([O.sin(x)]))[0] ^ 0x80000000
        assert O.cos(-x) == O.cos(x)


@pytest.mark.parametrize("radius", [0.1, 0.3, 0.5])
def test_rule_against_host_libm_on_clouds(radius):
    """the statement in both trig modes on the 58 k ROI cloud: the share of points whose bits differ is reported; on
    points whose smallest eigenvalue is well separated the normals agree within 1e-3 rad and the curvatures to 1e-3"""
    c = K.roi_cloud(7, 64, 2048)
    a, cnt, _, roots = O.normals(c, radius, details=True)
    b = O.normals(c, radius, trig_mode=1)
    ok = ~np.isnan(a[:, 0]) & ~np.isnan(b[:, 0])
    diff = (bits(a) != bits(b)).any(axis=1)
    print("\nradius %.1f: %.3f %% of the points differ in some bit" % (radius, 100.0 * diff.mean()))
    gap = (roots[:, 1] - roots[:, 0]) / np.maximum(roots[:, 2], 1e-30)
    good = ok & (gap > 1e-2)
    cosang = np.abs((a[good, :3].astype(np.float64) * b[good, :3]).sum(1))
    assert np.arccos(np.minimum(cosang, 1.0)).max() < 1e-3
    # the curvature is lambda0 / trace: its error is bounded relative to its value, or to 1e-2 for nearly planar sets
    err = np.abs(a[good, 3].astype(np.float64) - b[good, 3]) / np.maximum(np.abs(a[good, 3]), 1e-2)
    assert err.max() < 1e-3
    assert diff.mean() < 0.2
