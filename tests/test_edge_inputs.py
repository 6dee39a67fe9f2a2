"""The edge-case generators (tests/edge_inputs.py) on the CPU: their inputs reach the fragile spots they are meant to reach,
and the two CPU references -- the C++ oracle and the numpy restatement -- agree on every one of them."""
import numpy as np
import pytest

import edge_inputs as E
from helpers import cloud_dict
from oracle import np_oracle

F32 = np.float32


@pytest.mark.parametrize("leaf", E.LEAVES)
def test_lattice_points_discriminate_the_cell_formula(leaf):
    """A kernel that computed x / leaf, or rounded the product x * inv towards zero, must misplace some lattice points: at
    least 2 % of their coordinates fall into another cell under either formula. Power-of-two leaves have exact products --
    no formula can differ there -- and their planes k * leaf are exact, so x0 lies on the plane and x0 - 1 ulp below it."""
    x = E.lattice_cloud(11, leaf)[:, :3]
    d = E.lattice_discrimination(leaf, x)
    if float(np.log2(leaf)).is_integer():
        assert d["either"] == 0.0
        v = E.lattice_values(leaf, np.arange(-5, 6))
        x0, below = v[:11], v[11 * 2:11 * 3]     # x0, then +1 ulp, then -1 ulp
        assert (np.floor(x0 * E.inv_of(leaf)) == np.arange(-5, 6)).all()
        assert (np.floor(below * E.inv_of(leaf)) == np.arange(-5, 6) - 1).all()
    else:
        assert d["vs_division"] >= 0.02 and d["vs_round_to_zero"] >= 0.015, d
    assert (x < 0).any() and (x > 0).any() and (x == 0).any()


def test_box_limit_points_land_on_the_limits():
    """Family B: after the unfused transform the box limits, and one ulp either side of each, occur in the data."""
    t = (1.25, 0.5, 0.375)
    box = [(-2.5, 7.25), (-3.0, 3.5), (-1.5, 2.0)]
    x = E.box_limit_cloud(5, t, box, intensity_window=(10.0, 200.0))
    y = np_oracle.transform(x, E.identity_extrinsic(t)[:3].reshape(-1))
    for a in range(3):
        for v in E.limit_values(*box[a]):
            assert (y[:, a] == v).sum() >= 3, (a, v)
    for v in E.limit_values(10.0, 200.0):
        assert (y[:, 3] == v).sum() >= 3


def test_signed_zero_and_subnormals_survive_the_transform():
    x = E.signed_zero_subnormal_cloud(3)
    y = np_oracle.transform(x, E.identity_extrinsic((-0.0, -0.0, -0.0)).reshape(-1))
    special = (np.abs(x[:, :3]) < np.finfo(F32).tiny).any(axis=1) | (np.abs(x[:, 3]) < np.finfo(F32).tiny)
    assert (y[special].view(np.uint32) == x[special].view(np.uint32)).all(), "-0.0 and subnormals must keep every bit"
    sub = (np.abs(y[:, :3]) > 0) & (np.abs(y[:, :3]) < np.finfo(F32).tiny)
    assert sub.any(axis=0).all() and (np.signbit(y[:, :3]) & (y[:, :3] == 0)).any(axis=0).all()


@pytest.mark.parametrize("div,overflow,bits", [(E.DIV_2P31, True, 31), (E.DIV_2P31_PLUS, True, 32), (E.DIV_2P32, True, 32),
                                               (E.DIV_2P32_PLUS, True, 33), (E.DIV_GUARD_BELOW, False, 31),
                                               (E.DIV_GUARD_ABOVE, True, 32)])
def test_grid_cloud_has_the_intended_grid(oracle, div, overflow, bits):
    x = E.grid_cloud(1, div, n_filler=2000)
    o = oracle.voxelgrid(x, [1.0] * 3, 1, True, force64=True)
    assert o["div_b"].tolist() == list(div) and o["pcl_overflow"] == overflow
    assert E.bits_for(int(np.prod(np.asarray(div, np.int64)))) == bits


def test_guard_and_key_grid_disagree(oracle):
    """Points at 0.9 and a - 0.9: PCL's d is a - 1 per axis, the key grid a cells. At a = 1291 the guard passes
    (1290^3 <= INT32_MAX) while the grid holds more than INT32_MAX cells."""
    x = E.grid_cloud(2, E.DIV_GUARD_ABOVE, n_filler=2000, inset=0.9)
    o = oracle.voxelgrid(x, [1.0] * 3, 1, True, force64=True)
    assert o["div_b"].tolist() == list(E.DIV_GUARD_ABOVE) and not o["pcl_overflow"]
    assert int(np.prod(o["div_b"].astype(np.int64))) > 2**31 - 1


# ---- the two references on every family --------------------------------------------------------------------------------
def edge_cases():
    """(name, clouds [(xyzi, m, is_dense)], passes, leaf) -- the frames the GPU edge tests run, small enough for the CPU."""
    cases = []
    for leaf in E.LEAVES:
        x = E.lattice_cloud(100, leaf, n_lattice=6000, n_filler=3000)
        cases.append(("A-leaf%g" % leaf, [(x, E.identity_extrinsic((0, 0, 0)), 1)], [], leaf))
    t = (1.25, 0.5, 0.375)
    box = [(-2.5, 7.25), (-3.0, 3.5), (-1.5, 2.0)]
    for dense in (1, 0):
        x = E.box_limit_cloud(7, t, box, intensity_window=(10.0, 200.0))
        if not dense:
            x[::97, 1] = np.nan
        passes = [(a, box[a][0], box[a][1], 0) for a in range(3)]
        cases.append(("B-box-dense%d" % dense, [(x, E.identity_extrinsic(t), dense)], passes, 0.25))
        cases.append(("B-box-int-dense%d" % dense, [(x, E.identity_extrinsic(t), dense)], passes + [(3, 10.0, 200.0, 0)], 0.1))
    m = E.rotated_extrinsic(0.7, (3.0, -2.0, 1.5), pitch=0.05)
    x = E.lattice_cloud(8, 0.1, n_lattice=4000, n_filler=4000)
    lim = E.limits_from_data(np_oracle.transform(x, m.reshape(-1)))
    cases.append(("B-rotated", [(x, m, 1)], [(a, lo, hi, 0) for a, lo, hi in lim], 0.1))
    z = E.signed_zero_subnormal_cloud(9)
    mz = E.identity_extrinsic((-0.0, -0.0, -0.0))
    for lo, hi in ((0.0, 0.5), (-0.5, 0.0)):
        cases.append(("B-zero-%g-%g" % (lo, hi), [(z, mz, 1)], [(a, lo if a == 0 else -1.0, hi if a == 0 else 1.0, 0)
                                                                  for a in range(3)] + [(3, 0.0, 255.0, 0)], 0.05))
    for leaf in (0.02, 0.05, 0.1):
        x = E.offset_cloud(20, leaf, n=12000)
        cases.append(("C-map-leaf%g" % leaf, [(x, E.identity_extrinsic((0, 0, 0)), 1)], [], leaf))
    xs = E.lattice_cloud(21, 0.05, n_lattice=5000, n_filler=5000)
    mk = E.rotated_extrinsic(-1.1, (2500.0, -3800.0, 35.0))
    cases.append(("C-km-extrinsic", [(xs, mk, 1)], [(2, 30.0, 40.0, 0)], 0.05))
    for div in (E.DIV_2P31, E.DIV_2P31_PLUS, E.DIV_GUARD_BELOW, E.DIV_GUARD_ABOVE):
        cases.append(("D-%s" % "x".join(map(str, div)), [(E.grid_cloud(3, div, n_filler=4000), E.identity_extrinsic((0, 0, 0)), 1)],
                      [], 1.0))
    cases.append(("D-guard-disagrees", [(E.grid_cloud(4, E.DIV_GUARD_ABOVE, n_filler=4000, inset=0.9),
                                         E.identity_extrinsic((0, 0, 0)), 1)], [], 1.0))
    return cases


CASES = edge_cases()


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("min_points", [1, 2])
def test_oracles_agree_on_edge_inputs(oracle, case, min_points):
    name, clouds, passes, leaf = case
    cds = [cloud_dict(x, m, dense) for x, m, dense in clouds]
    c = oracle.merge_frame(cds, passes, [leaf] * 3, min_points, True, True)
    n = np_oracle.merge_frame(cds, passes, [leaf] * 3, min_points, True, True)
    assert c["n_survivors"] == len(n["survivor_src"]) > 0
    assert (c["survivor_src"] == n["survivor_src"]).all()
    assert (c["survivor_xyzi"].view(np.uint32) == n["survivor_xyzi"].view(np.uint32)).all()
    v = n["voxel"]
    assert c["min_b"].tolist() == v["min_b"].tolist() and c["div_b"].tolist() == v["div_b"].tolist()
    assert c["pcl_overflow"] == v["pcl_overflow"]
    assert (c["point_idx"] == v["point_idx"]).all(), "voxel membership"
    assert (c["idx"] == v["idx"]).all() and (c["count"] == v["count"]).all()
    np.testing.assert_allclose(c["centroid_f64"], v["centroid_f64"], rtol=1e-12, atol=1e-12)
    assert c["n_voxels"] > 0
