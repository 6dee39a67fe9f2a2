"""CPU checks of the zone slicing's edge inputs (tests/zone_edges.py, family Z): the restated constants match
cm_zones.cu, the cases land where they were built (membership flips on warp-row and tile edges, points in 0, 1, several
and all zones, zone 15 alone, every zone present in every scan round), the no-op stage changes nothing in either oracle,
the two oracles agree (including NaN limits, where PassThrough keeps every finite value), and the zone total's sum is
64-bit in the source."""
import os
import re

import numpy as np
import pytest

import zone_edges as Z
from oracle import np_oracle as npo

SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "cloud_merger_b200", "csrc")
INC = os.path.join(os.path.dirname(SRC), "..", "include", "cloud_merger_gpu.h")
F32 = np.float32


def _src(name):
    with open(os.path.join(SRC, name)) as f:
        return f.read()


def test_zone_constants_match_the_source():
    zn = _src("cm_zones.cu")
    assert "constexpr int ZN_THREADS = 256;" in zn and "constexpr int ZN_IPT = 4;" in zn
    assert "constexpr int ZN_TILE = ZN_THREADS * ZN_IPT;" in zn and Z.ZN_TILE == 256 * 4
    assert "warp * (32 * ZN_IPT) + lane" in zn and Z.WARP_ROW == 32 * 4
    assert "i0 += 1024u * 8u" in zn and "k_zone_scan<<<p.zones.n_zones, 1024, 0, stream>>>" in zn
    assert Z.SCAN_TILES == 1024 * 8 and Z.SCAN_POINTS == Z.SCAN_TILES * Z.ZN_TILE
    assert "uint32_t run = s_run + s_scr[w] + incl - sum;" in zn and "if (tid == 0) s_run += s_scr[32];" in zn
    assert re.search(r"#define CM_MAX_ZONES (\d+)", open(INC).read()).group(1) == str(Z.MAX_ZONES)
    # the zones' total: a 64-bit sum, saturated past 0xFFFFFFF0 so that the host does not regrow
    assert "unsigned long long run = 0;" in zn and "run > 0xFFFFFFF0ull ? 0xFFFFFFFFu : (uint32_t)run" in zn
    assert "if (run > p.out_capacity) *p.overflow = total;" in zn
    assert "(size_t)report[CM_MAX_ZONES + 1] <= 0xFFFFFFF0u" in _src("cm_api.cu")
    # the box test skips the intensity for zones without an intensity stage
    assert "(no_i_mask >> z)" in zn


@pytest.mark.parametrize("n", Z.TILE_NS)
def test_tile_cases_land_on_the_edges(n):
    for case in Z.tile_cases():
        if case["name"] != "Z-tile:%d" % n:
            continue
        m = Z.np_zone_masks(case["x"], case["zones"])
        per = m.sum(axis=0)
        if n >= 32:
            assert 0 in per and 1 in per and (per >= 3).any()
        for edge in (Z.WARP_ROW, Z.ZN_TILE):   # some zone changes membership across the edge
            if n > edge:
                assert (m[:, edge - 1] != m[:, edge]).any(), edge
    x = Z._index_cloud(n, n)
    only = Z.np_zone_masks(x, Z.ONLY_15)
    assert not only[:15].any() and only[15].any()
    per = Z.np_zone_masks(x, Z.NESTED).sum(axis=0)
    if n > 1024:
        assert Z.MAX_ZONES in per and 1 in per and 0 in per
        assert per[1023] == 15 and per[1024] == 16 and per[127] == 1 and per[128] == 2


def test_scan_cases_fill_every_round():
    for n in Z.SCAN_NS:
        m = Z.np_zone_masks(Z.scan_cloud(n), Z.SCAN_ZONES)
        rounds = (n + Z.SCAN_POINTS - 1) // Z.SCAN_POINTS
        assert rounds >= 2
        for r in range(rounds):
            a, b = r * Z.SCAN_POINTS, min(n, (r + 1) * Z.SCAN_POINTS)
            assert m[:, a:b].any(axis=1).all(), r
        assert m.sum() <= 2 * n   # fits the outputs sized for twice the input: no regrow


@pytest.mark.parametrize("name", sorted(Z.PATH_SETS))
def test_noop_stage_and_oracles_agree(oracle, name):
    x = Z.path_cloud()
    zones = Z.PATH_SETS[name]
    forced = Z.with_noop(zones)
    assert not Z.is_box(forced)
    m = Z.np_zone_masks(x, zones)
    assert (Z.np_zone_masks(x, forced) == m).all()
    a, b = oracle.zone_split(x, zones), oracle.zone_split(x, forced)
    for k, ((ax, ai), (bx, bi)) in enumerate(zip(a, b)):
        assert (ai == bi).all() and ax.tobytes() == bx.tobytes()
        assert (ai.astype(np.int64) == np.nonzero(m[k])[0]).all(), (name, k)


def test_tile_cases_oracles_agree(oracle):
    for case in Z.tile_cases():
        m = Z.np_zone_masks(case["x"], case["zones"])
        for k, (_, src) in enumerate(oracle.zone_split(case["x"], case["zones"])):
            assert (src.astype(np.int64) == np.nonzero(m[k])[0]).all(), (case["name"], k)


def test_nan_limit_keeps_every_finite_value(oracle):
    """PCL drops a point when `v < lo || v > hi` (negative: `v >= lo && v <= hi`): a NaN limit tests nothing on its
    side, and a negative window with a NaN limit drops nothing. The numpy PassThrough used to keep nothing there."""
    x = Z.path_cloud()
    fin = np.isfinite(x[:, :3]).all(axis=1)
    for neg in (0, 1):
        for lo, hi in ((float("nan"), 1.0), (0.0, float("nan")), (float("nan"), float("nan"))):
            want = oracle.passthrough(x, 0, lo, hi, bool(neg))
            got = np.nonzero(npo.passthrough_mask(x, 0, lo, hi, bool(neg)))[0]
            assert len(got) == len(want) and (got == want).all(), (lo, hi, neg)
            if neg or lo != lo and hi != hi:
                assert (got == np.nonzero(fin)[0]).all()
