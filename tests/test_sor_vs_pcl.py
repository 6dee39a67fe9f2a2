"""The C++ statistical-outlier-removal statement (tests/sor_oracle.cpp) against the REAL pcl::StatisticalOutlierRemoval
(tests/sor_pcl_ref.cpp) on the clouds of the CPU tests and the known answers. Where PCL is not installed (this repository's
build image) these tests SKIP and say why; where pkg-config finds PCL >= 1.8 the wrapper is built on first use. The sqrt
reading of the installed build is found by trying both."""
import json
import os

import numpy as np
import pytest

import sor_cases as K
import sor_oracle as O

pytestmark = pytest.mark.skipif(not O.pcl_available(), reason="real-PCL StatisticalOutlierRemoval not available: " + O.pcl_why_not())


@pytest.mark.parametrize("mean_k,std_mul,negative", [(1, 1.0, False), (8, 0.0, True), (30, 2.0, False)])
def test_survivors_match_pcl(mean_k, std_mul, negative):
    clouds = [K.blobs(3, 1200), K.with_duplicates(K.blobs(4, 800), 4, 0.5), K.lattice(7),
              K.with_nonfinite(K.blobs(5, 900), 5, 0.1)]
    for x in clouds:
        want = O.pcl_statistical_outlier(x, mean_k, std_mul, negative)
        got = [np.nonzero(O.statistical_outlier(x, mean_k, std_mul, negative, m)["keep"])[0] for m in (0, 1)]
        assert any(np.array_equal(g, want) for g in got)


def test_known_answers():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sor.json")) as f:
        cases = json.load(f)
    for c in cases:
        if c["too_few"]:
            continue  # PCL's behaviour there is undefined
        pts = np.array([int(h, 16) for row in c["xyzi"] for h in row], np.uint32).view(np.float32).reshape(-1, 4)
        got = O.pcl_statistical_outlier(pts, c["mean_k"], c["std_mul"], bool(c["negative"]))
        assert got.tolist() == c["kept"], c["name"]
