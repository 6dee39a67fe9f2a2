"""The C++ statement of PCL's cluster loop (tests/ec_oracle.cpp) against the REAL pcl::EuclideanClusterExtraction
(tests/ec_pcl_ref.cpp) on finite clouds of the CPU tests and the golden answers. Where PCL is not installed (this
repository's build image) these tests SKIP and say why; where pkg-config finds PCL >= 1.8 the wrapper is built on first
use. The cluster order compared is that of a GCC (libstdc++) build of PCL."""
import json
import os

import numpy as np
import pytest

import ec_cases as K
import ec_oracle as O

pytestmark = pytest.mark.skipif(not O.pcl_available(), reason="real-PCL EuclideanClusterExtraction not available: " +
                                O.pcl_why_not())


def _same(a, b):
    return len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("tolerance,min_size,max_size", [(0.5, 1, O.INT_MAX), (0.3, 3, 50), (0.1, 1, O.INT_MAX)])
def test_clusters_match_pcl(tolerance, min_size, max_size):
    clouds = [K.blobs(3, 1200), K.with_duplicates(K.lattice(8, 0.25), 4, 0.5), K.lattice(7, 0.5),
              K.equal_clusters(5, 40, 5, 0.5), K.ulp_pairs(6, tolerance)]
    for x in clouds:
        assert _same(O.euclidean_clusters(x, tolerance, min_size, max_size),
                     O.pcl_euclidean_clusters(x, tolerance, min_size, max_size))


def test_golden_answers():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ec.json")) as f:
        cases = json.load(f)["cases"]
    for c in cases:
        pts = np.array([[float(v) for v in r] for r in c["xyzi"]], np.float32).reshape(-1, 4)
        if not np.isfinite(pts[:, :3]).all():
            continue  # PCL searches from non-finite points (a documented deviation)
        got = O.pcl_euclidean_clusters(pts, c["tolerance"], c["min_size"], c["max_size"])
        assert [g.tolist() for g in got] == c["clusters"], c["name"]
