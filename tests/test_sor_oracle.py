"""CPU tests of the pcl::StatisticalOutlierRemoval statements (not gpu): the C++ oracle (tests/sor_oracle.cpp), the numpy
restatement (tests/sor_np.py) and the known answers of tests/golden/sor.json (worked out step by step) agree bit for bit on
per-point distances, statistics and survivors; the new C-ABI symbols are exported and the new structs have the layout of
their ctypes mirrors."""
import ctypes as C
import json
import os
import subprocess
import tempfile

import numpy as np
import pytest

import sor_cases as K
import sor_np
from sor_oracle import statistical_outlier

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _golden():
    with open(os.path.join(ROOT, "tests", "golden", "sor.json")) as f:
        return json.load(f)


def _f32(hexes):
    return np.array([int(h, 16) for h in hexes], np.uint32).view(np.float32)


def _f64(h):
    return np.array([int(h, 16)], np.uint64).view(np.float64)[0]


def _bits_equal(a, b):
    a, b = np.float64(a), np.float64(b)
    return (np.isnan(a) and np.isnan(b)) or a.tobytes() == b.tobytes()


def assert_same(got, want, what):
    assert np.array_equal(np.asarray(got["distances"], np.float32).view(np.uint32),
                          np.asarray(want["distances"], np.float32).view(np.uint32)), what
    assert np.array_equal(np.nonzero(got["keep"])[0], np.nonzero(want["keep"])[0]), what
    assert got["n_valid"] == want["n_valid"] and got["too_few"] == want["too_few"], what
    for k in ("mean", "stddev", "threshold"):
        assert _bits_equal(got[k], want[k]), (what, k, got[k], want[k])


@pytest.mark.parametrize("case", [c["name"] for c in _golden()])
def test_golden_known_answers(case):
    c = next(c for c in _golden() if c["name"] == case)
    pts = _f32([h for row in c["xyzi"] for h in row]).reshape(-1, 4)
    keep = np.zeros(len(pts), bool)
    keep[c["kept"]] = True
    want = {"distances": _f32(c["distances"]), "keep": keep, "n_valid": c["n_valid"], "too_few": c["too_few"],
            "mean": _f64(c["mean"]), "stddev": _f64(c["stddev"]), "threshold": _f64(c["threshold"])}
    args = (c["mean_k"], c["std_mul"], bool(c["negative"]), c["sqrt_mode"])
    assert_same(statistical_outlier(pts, *args), want, "C++ oracle")
    assert_same(sor_np.sor_cloud(pts, *args), want, "numpy restatement")


def _clouds():
    lat = K.lattice(7)
    off = K.blobs(12, 900, spread=2.0)
    off[:, 0] = (off[:, 0] + np.float32(5.0e5)).astype(np.float32)
    nan_step = next(s for s in np.linspace(0.1, 0.3, 200, dtype=np.float32)
                    if np.isnan(sor_np.sor_cloud(K.lattice(6, float(s)), 1, 1.0)["threshold"]))
    return {"blobs": K.blobs(3, 1200), "duplicates": K.with_duplicates(K.blobs(4, 800), 4, 0.5), "lattice": lat,
            "nonfinite": K.with_nonfinite(K.blobs(5, 900), 5, 0.1), "utm": off, "faces": K.shell_faces(6, 0.3, 200),
            "nan_threshold": K.lattice(6, float(nan_step)), "too_few": K.with_nonfinite(K.blobs(7, 5, outliers=0), 7, 0.4)}


@pytest.mark.parametrize("name", sorted(_clouds()))
@pytest.mark.parametrize("mean_k,std_mul,negative,sqrt_mode", [(1, 1.0, False, 0), (6, 0.0, True, 1), (18, 2.0, False, 1),
                                                               (50, -0.5, False, 0)])
def test_oracle_and_numpy_agree(name, mean_k, std_mul, negative, sqrt_mode):
    x = _clouds()[name]
    a = statistical_outlier(x, mean_k, std_mul, negative, sqrt_mode)
    b = sor_np.sor_cloud(x, mean_k, std_mul, negative, sqrt_mode)
    assert_same(a, b, name)
    if name == "nan_threshold" and mean_k == 1:
        assert np.isnan(a["threshold"]) and a["keep"].all()


def test_sqrt_modes_differ_somewhere():
    """the two sqrt readings of PCL's loop are not the same function: on an ordinary cloud some distances differ"""
    x = K.blobs(8, 1500)
    a = sor_np.sor_cloud(x, 10, 1.0, False, 0)["distances"]
    b = sor_np.sor_cloud(x, 10, 1.0, False, 1)["distances"]
    assert (a != b).any()


def test_abi_symbols_and_struct_sizes():
    from cloud_merger_b200 import _lib
    lib = _lib.load()
    for n in ("cm_dev_statistical_outlier", "cm_dev_statistical_outlier_multi", "cm_statistical_outlier",
              "cm_statistical_outlier_multi", "cm_get_statistical_out"):
        assert n in _lib.SYMBOLS and hasattr(lib, n), n
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "cloud_merger_gpu.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %d %d %d\n", sizeof(cm_sor_cfg_t), sizeof(cm_sor_stats_t), sizeof(cm_sor_out_t),
         offsetof(cm_sor_cfg_t, std_mul), offsetof(cm_sor_out_t, cloud), CM_SOR_MAX_K, CM_SOR_SQRT_DOUBLE,
         CM_SOR_SQ_SUM_SERIAL);
  return 0;
}'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(v) for v in subprocess.check_output([exe]).split()]
    assert got == [C.sizeof(_lib.CmSorCfg), C.sizeof(_lib.CmSorStats), C.sizeof(_lib.CmSorOut),
                   _lib.CmSorCfg.std_mul.offset, _lib.CmSorOut.cloud.offset, _lib.CM_SOR_MAX_K, _lib.CM_SOR_SQRT_DOUBLE,
                   _lib.CM_SOR_SQ_SUM_SERIAL]
