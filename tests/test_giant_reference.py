"""CPU tests of the giant-cloud partition reference (tests/giant_reference.py) and of the giant-cloud edge inputs: the
reference against hand-computed plans and against the torch formulation of the host protocol (multi_gpu), and the edge
clouds against the targets they are built for."""
import numpy as np
import pytest
import torch

import edge_inputs as E
import giant_reference as R
from cloud_merger_b200 import multi_gpu

WORLDS = (2, 3, 4, 8, 16)
ALL_CASES = [c + s for c in list(E.GIANT_CASES) + list(E.GIANT_RANGE_CASES) for s in ("", "+nf")]
U64 = (1 << 64) - 1


@pytest.mark.parametrize("case", ALL_CASES)
def test_reference_agrees_with_the_host_protocol(case):
    """Grid, keys and splitters of the reference against multi_gpu.global_grid / voxel_keys / pick_splitters on CPU
    tensors (the torch formulation the gloo tests run), for every edge cloud and every rank count."""
    x, leaf = E.giant_case(case)
    g = R.grid(x, leaf)
    if g["finite"] == 0:   # the torch formulation has no grid for a cloud without finite points
        assert g["cells"] == 1 and g["key_bits"] == 0 and not g["key_range_error"]
        return
    t = torch.from_numpy(x)
    mn, mx, min_b, div_b = multi_gpu.global_grid(t, [leaf] * 3)
    assert (mn.view(np.uint32) == g["min_p"].view(np.uint32)).all() and (mx.view(np.uint32) == g["max_p"].view(np.uint32)).all()
    assert min_b.tolist() == g["min_b"].tolist() and div_b.tolist() == g["div_b"].tolist()
    if g["key_range_error"]:
        return
    k = R.keys(x, leaf, g["min_b"], g["div_b"])
    tk = multi_gpu.voxel_keys(t, [leaf] * 3, min_b, div_b).numpy()
    assert (tk == k).all()
    assert k.max() < g["cells"] and (k[R.finite_rows(x)] >= 0).all()
    width = R.bin_width(g["cells"])
    h = R.histogram(k, g["cells"])
    for w in WORLDS:
        want = multi_gpu.pick_splitters(torch.from_numpy(tk), g["cells"], w, bins=R.BINS).tolist()
        assert R.splitters(h, width, w) == [v & U64 for v in want], w


def test_three_finite_points_over_eight_ranks():
    x = np.array([[0.5, 0.5, 0.5, 1], [np.nan, 0, 0, 2], [2.5, 0.5, 0.5, 3], [1.5, 1.5, 0.5, 4], [0, np.inf, 0, 5]], np.float32)
    p = R.plan(x, 1.0, 8, me=3)
    assert p["min_b"].tolist() == [0, 0, 0] and p["div_b"].tolist() == [3, 2, 1] and p["cells"] == 6 and p["key_bits"] == 3
    assert p["keys"].tolist() == [0, -1, 2, 4, -1] and p["width"] == 1 and p["total"] == 3
    # targets 3r//8 = 0 0 1 1 1 2 2; running sums 1 1 2 2 3 (bins 0..4)
    assert p["splitters"] == [1, 1, 1, 1, 1, 3, 3]
    assert p["dest"].tolist() == [0, 3, 5, 7, 3]
    assert [q.tolist() for q in p["parts"]] == [[0], [], [], [1, 4], [], [2], [], [3]]
    assert p["send_begin"] == [0, 1, 1, 1, 3, 3, 4, 4, 5] and p["points_sent_away"] == 3


def test_one_voxel_and_empty_clouds():
    x = np.full((10, 4), 0.25, np.float32)
    x[:, 0] = np.linspace(0.01, 0.99, 10).astype(np.float32)
    p = R.plan(x, 1.0, 4, me=2)
    assert p["cells"] == 1 and p["key_bits"] == 0 and p["width"] == 1 and (p["keys"] == 0).all()
    assert p["splitters"] == [1, 1, 1] and (p["dest"] == 0).all() and p["points_sent_away"] == 10
    for e in (np.zeros((0, 4), np.float32), np.full((6, 4), np.nan, np.float32)):
        p = R.plan(e, 0.1, 5, me=4)
        assert p["splitters"] == [1, 1, 1, 1] and p["total"] == 0 and p["key_bits"] == 0
        assert p["send_begin"] == [0, 0, 0, 0, 0, len(e)] and p["points_sent_away"] == 0


def test_negative_cells_and_key_range():
    x = np.array([[-0.5, -1.0, 0.0, 0], [0.5, -0.999, 1.0, 0]], np.float32)
    g = R.grid(x, 1.0)
    assert g["min_b"].tolist() == [-1, -1, 0] and g["div_b"].tolist() == [2, 1, 2]
    assert R.keys(x, 1.0, g["min_b"], g["div_b"]).tolist() == [0, 3]
    assert R.grid(E.giant_case("axis:2p21")[0], 1.0)["key_range_error"] is False
    assert R.grid(E.giant_case("origin:ok+")[0], 1.0)["key_range_error"] is False
    for c in E.GIANT_RANGE_CASES:
        assert R.grid(E.giant_case(c)[0], 1.0)["key_range_error"] is True, c


@pytest.mark.parametrize("bits", sorted(E.KEY_WIDTH_DIVS))
def test_key_width_clouds_hit_their_width(bits):
    x, leaf = E.giant_case("bits:%d" % bits)
    g = R.grid(x, leaf)
    assert g["div_b"].tolist() == list(E.KEY_WIDTH_DIVS[bits]) and g["key_bits"] == bits and not g["key_range_error"]
    xn, _ = E.giant_case("bits:%d+nf" % bits)
    fin = R.finite_rows(xn)
    assert (xn[fin].view(np.uint32) == x.view(np.uint32)).all(), "the non-finite variant keeps the finite rows in order"
    assert (~fin).sum() >= len(x) // 500 + 3 and np.isnan(xn[:, :3]).any() and np.isinf(xn[:, :3]).any()


@pytest.mark.parametrize("wname", sorted(E.BIN_WIDTH_DIVS))
def test_bin_boundary_clouds_decide_the_splitters(wname):
    """The points sit exactly on the keys k*width - 1 / k*width / k*width + 1, and moving one count across any of those bin
    boundaries, either way, changes a splitter for some rank count."""
    div = E.BIN_WIDTH_DIVS[wname]
    x, leaf = E.giant_case("bin:" + wname)
    g = R.grid(x, leaf)
    assert g["min_b"].tolist() == [0, 0, 0] and g["div_b"].tolist() == list(div)
    width = R.bin_width(g["cells"])
    assert width == {"w1": 1, "w64": 64, "w63": 63, "w2p40": (1 << 40) + (1 << 28)}[wname]
    k = R.keys(x, leaf, g["min_b"], g["div_b"])
    want = E.grid_corner_keys(div) + E.bin_boundary_keys(div)
    assert k.tolist() == want
    h = R.histogram(k, g["cells"])
    base = {w: R.splitters(h, width, w) for w in WORLDS}
    for kb in (R.BINS // 4, R.BINS // 2, 3 * R.BINS // 4):
        assert (kb * width - 1) // width == kb - 1 and (kb * width) // width == kb
        for src, dst in ((kb - 1, kb), (kb, kb - 1)):
            assert h[src] > 0
            moved = h.copy()
            moved[src] -= 1
            moved[dst] += 1
            assert any(R.splitters(moved, width, w) != base[w] for w in WORLDS), (kb, src, dst)


@pytest.mark.parametrize("kind", E.DEGENERATE_KINDS)
def test_degenerate_clouds(kind):
    x, leaf = E.giant_case("deg:" + kind)
    g = R.grid(x, leaf)
    fin = int(R.finite_rows(x).sum())
    want = {"empty": (0, 0), "all-nonfinite": (0, len(x)), "one-point": (1, 1), "one-voxel": (len(x), len(x)),
            "three-finite": (3, len(x)), "hot-voxel": (len(x), len(x))}[kind]
    assert (fin, len(x)) == want
    if kind in ("one-voxel", "one-point"):
        assert g["cells"] == 1
    if kind == "hot-voxel":   # several balancing targets of 16 ranks in one histogram bin: some ranks get nothing
        p = R.plan(x, leaf, 16)
        assert len(set(p["splitters"])) < 15 and min(len(q) for q in p["parts"]) == 0


@pytest.mark.parametrize("bits", sorted(E.KEY_WIDTH_DIVS))
def test_oracles_agree_on_the_key_width_grids(oracle, bits):
    """The C++ oracle and its numpy restatement on the key-width grids: the same voxels, and the same PCL guard -- also at
    2^21 cells on every axis, where the product of the cell counts is 2^63."""
    from oracle import np_oracle
    x, leaf = E.giant_case("bits:%d" % bits)
    a = oracle.voxelgrid(x, [leaf] * 3, 1, True, force64=True)
    b = np_oracle.voxelgrid(x, [leaf] * 3, 1, True, True)
    assert a["pcl_overflow"] == b["pcl_overflow"] == (int(np.prod(np.asarray(E.KEY_WIDTH_DIVS[bits], np.float64))) > 2**31 - 1)
    assert (a["idx"] == b["idx"]).all() and (a["count"] == b["count"]).all()
