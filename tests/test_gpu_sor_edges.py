"""GPU parity (-m gpu) of the statistical outlier removal at its edges (tests/sor_edges.py, family S): the register-slot
layouts, the stopping bound past every growth step near the origin and at |x * inv| ~ 2^19, the key plan (widths, pass
counts, the sentinel frame, the table limit, the floor and the clamps), the two sums at their exactness boundary, and
distances on the threshold. Every case runs through the four entry points (host and device, single and multi), with the
table and with the binary searches where the table applies; per-point distances, per-cloud statistics and sum path, and
the survivors must be bit-exact against tests/sor_np.py, and cm_launch_count must equal sor_plan's count."""
import numpy as np
import pytest

import sor_edges as S
import sor_np
from cloud_merger_b200 import CloudMerger
from helpers import assert_bit_equal

pytestmark = pytest.mark.gpu

CASES = S.sor_cases()
CAP = 1 << 14


@pytest.fixture(scope="module")
def cm(gpu_ok):
    with CloudMerger(max_sensors=1, max_points_per_sensor=CAP, max_batch_points=CAP, max_batch_frames=16) as m:
        yield m


def _same(a, b):
    return (np.isnan(a) and np.isnan(b)) or np.float64(a).tobytes() == np.float64(b).tobytes()


def _compare(out, got, clouds, want, begin, force_serial, what):
    assert len(out["clouds"]) == len(clouds), what
    for c, (cloud, w, (gx, gi)) in enumerate(zip(clouds, want, got)):
        wc = "%s, cloud %d" % (what, c)
        assert_bit_equal(out["distances"][begin[c]:begin[c + 1]], w["distances"], "distances of " + wc)
        st = out["clouds"][c]
        assert st["n_valid"] == w["n_valid"] and st["too_few"] == w["too_few"], (wc, st, w["n_valid"])
        assert st["sum_path"] == S.sum_path(w["distances"], force_serial), (wc, st["sum_path"])
        if not w["too_few"]:
            for k in ("mean", "stddev", "threshold"):
                assert _same(st[k], w[k]), (wc, k, st[k], w[k])
        keep = np.nonzero(w["keep"])[0]
        assert len(gi) == len(keep) and (gi.astype(np.int64) == keep).all(), "survivor set / order of " + wc
        assert_bit_equal(gx, cloud[keep], "survivor coordinates of " + wc)


def run_four(cm, clouds, mean_k, std_mul, negative, sqrt_mode, launches, force_serial, what):
    want = sor_np.sor(clouds, mean_k, std_mul, negative, sqrt_mode)
    begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    buf = cm.upload(np.ascontiguousarray(np.concatenate(clouds)))
    got = cm.statistical_outlier_multi(clouds, mean_k, std_mul, negative, sqrt_mode)
    assert cm.launch_count() == launches, what + " (multi)"
    _compare(cm.statistical_outlier_out(), got, clouds, want, begin, force_serial, what + " (multi)")
    cm.dev_statistical_outlier_multi(buf.ptr, begin, mean_k, std_mul, negative, sqrt_mode)
    assert cm.launch_count() == launches, what + " (device multi)"
    got = [(x, (i.astype(np.int64) - begin[c]).astype(np.uint32)) for c, (x, i) in enumerate(cm.zone_out())]
    _compare(cm.statistical_outlier_out(), got, clouds, want, begin, force_serial, what + " (device multi)")
    if len(clouds) == 1:
        got = [cm.statistical_outlier(clouds[0], mean_k, std_mul, negative, sqrt_mode)]
        assert cm.launch_count() == launches, what + " (single)"
        _compare(cm.statistical_outlier_out(), got, clouds, want, begin, force_serial, what + " (single)")
        cm.dev_statistical_outlier(buf.ptr, len(clouds[0]), mean_k, std_mul, negative, sqrt_mode)
        assert cm.launch_count() == launches, what + " (device single)"
        got = [cm.zone_out()[0]]
        _compare(cm.statistical_outlier_out(), got, clouds, want, begin, force_serial, what + " (device single)")


@pytest.mark.parametrize("name", sorted(CASES))
def test_sor_edges_bit_exact(cm, monkeypatch, name):
    case = CASES[name]
    clouds, mean_k = case["clouds"], case["mean_k"]
    if "cell" in case:
        monkeypatch.setenv("CM_SOR_CELL", repr(float(case["cell"])))
    else:
        monkeypatch.delenv("CM_SOR_CELL", raising=False)
    monkeypatch.delenv("CM_SOR_SERIAL_SUMS", raising=False)
    with_table = S.sor_plan(clouds, mean_k, case.get("cell"))["table"]
    for table in ((True, False) if with_table else (True,)):
        if table:
            monkeypatch.delenv("CM_SOR_NO_TABLE", raising=False)
        else:
            monkeypatch.setenv("CM_SOR_NO_TABLE", "1")
        launches = S.sor_plan(clouds, mean_k, case.get("cell"), table)["launches"]
        for serial in ((False, True) if case.get("serial_too") else (False,)):
            if serial:
                monkeypatch.setenv("CM_SOR_SERIAL_SUMS", "1")
            for sm in case.get("sqrt_modes", (0,)):
                for neg in ((False, True) if case.get("negative_too") else (False,)):
                    what = "%s table=%s serial=%s sqrt_mode=%d negative=%s" % (name, table, serial, sm, neg)
                    run_four(cm, clouds, mean_k, case.get("std_mul", 1.0), neg, sm, launches, serial, what)
            monkeypatch.delenv("CM_SOR_SERIAL_SUMS", raising=False)
    monkeypatch.delenv("CM_SOR_NO_TABLE", raising=False)
