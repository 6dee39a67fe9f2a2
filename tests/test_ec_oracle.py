"""CPU tests of the Euclidean cluster extraction's references (no GPU): the C++ statement of PCL's seed-queue loop
(tests/ec_oracle.cpp), the component restatement (tests/ec_np.py) and the hand-worked answers of tests/golden/ec.json
agree bit for bit; the components equal PCL's loop on duplicate-heavy, lattice and random clouds; the restated
libstdc++ std::sort reproduces the C++ one, including its unstable order of equal sizes."""
import json
import os

import numpy as np
import pytest

import ec_cases as K
import ec_np
import ec_oracle as O
from helpers import host_function

HERE = os.path.dirname(os.path.abspath(__file__))
F32 = np.float32


def _same(a, b):
    return len(a) == len(b) and all(len(x) == len(y) and (np.asarray(x) == np.asarray(y)).all() for x, y in zip(a, b))


def _golden():
    with open(os.path.join(HERE, "golden", "ec.json")) as f:
        cases = json.load(f)["cases"]
    for c in cases:
        c["xyzi"] = np.array([[float(v) for v in r] for r in c["xyzi"]], F32).reshape(-1, 4)
    return cases


@pytest.mark.parametrize("case", _golden(), ids=lambda c: c["name"])
def test_golden_answers(case):
    args = (case["xyzi"], case["tolerance"], case["min_size"], case["max_size"])
    want = [np.array(c, np.int64) for c in case["clusters"]]
    assert _same(O.euclidean_clusters(*args), want)
    assert _same(ec_np.clusters_of(*args), want)


def test_r2_is_the_double_square_of_the_narrowed_tolerance():
    assert ec_np.r2_of(0.5) == F32(0.25)
    assert ec_np.r2_of(0.1) == np.nextafter(F32(0.1 * 0.1), F32(1))  # one float above the radius removal's (float)0.01


CLOUDS = {
    "lattice_exact_steps": (lambda: K.lattice(9, 0.5), 0.5),
    "lattice_one_ulp_more": (lambda: K.lattice(9, 0.5), float(np.nextafter(F32(0.5), F32(1)))),
    "lattice_duplicates": (lambda: K.with_duplicates(K.lattice(8, 0.25), 5, 0.8), 0.25),
    "repeated_points": (lambda: np.repeat(K.blobs(7, 60, outliers=0), 5, axis=0), 0.05),
    "blob_duplicates": (lambda: K.with_duplicates(K.blobs(6, 2000), 6, 0.5), 0.3),
    "ulp_pairs": (lambda: K.ulp_pairs(2, 0.1), 0.1),
    "cell_faces": (lambda: K.shell_faces(11, float(F32(0.5) * F32(1.00390625))), 0.5),
    "snake": (lambda: K.snake(3, 0.5), 0.5),
    "non_finite": (lambda: K.with_nonfinite(K.blobs(9, 3000), 9, 0.05), 0.3),
}


@pytest.mark.parametrize("name", sorted(CLOUDS))
@pytest.mark.parametrize("min_size,max_size", [(1, O.INT_MAX), (3, 50), (0, 0), (5, 4)])
def test_components_equal_pcl_seed_queue(name, min_size, max_size):
    make, tol = CLOUDS[name]
    c = make()
    assert _same(O.euclidean_clusters(c, tol, min_size, max_size), ec_np.clusters_of(c, tol, min_size, max_size))


@pytest.mark.parametrize("n,size", [(17, 4), (20, 5), (40, 7), (1500, 3)])
def test_cluster_order_on_equal_sizes(n, size):
    """17+ equal sizes take introsort's partitioning path: the restated sort matches libstdc++, and the order is not the
    stable one (the sort is unstable, which is why it has to be reproduced rather than replaced)"""
    rng = np.random.default_rng(n)
    for sizes in ([size] * n, [size] * n + [size + 1, size - 1, 2 * size], list(rng.integers(1, 4, n))):
        want = O.pcl_cluster_order(sizes)
        got = ec_np.pcl_cluster_order(sizes)
        assert (got == want).all()
        stable = np.argsort(-np.asarray(sizes), kind="stable")
        if len(set(sizes)) < len(sizes):
            assert not (want == stable).all()


def test_cluster_order_heap_path():
    """a sequence that runs introsort out of depth (many equal keys after median-of-three) matches libstdc++ too"""
    rng = np.random.default_rng(3)
    for n in (33, 257, 4096):
        sizes = list(rng.integers(1, 3, n))
        assert (ec_np.pcl_cluster_order(sizes) == O.pcl_cluster_order(sizes)).all()


def test_equal_size_clusters_through_both_statements():
    c = K.equal_clusters(1500, 1500, 3, 0.5, extra=(4, 2, 3, 6))
    a = O.euclidean_clusters(c, 0.5)
    assert len(a) == 1504 and _same(a, ec_np.clusters_of(c, 0.5))


def test_host_order_is_libstdcxx_sort_on_the_shared_cell_front_end():
    src = host_function("euclidean_clusters_run")
    assert 'radius_cell_keys(h, vp, tf, "CM_EC_NO_TABLE", table, st)' in src
    assert "ep.r2 = (float)((double)tf * (double)tf);" in src
    assert "const float cell = radius_f * 1.00390625f;" in host_function("radius_cell_keys")
    with open(os.path.join(os.path.dirname(HERE), "cloud_merger_b200", "csrc", "cm_api.cu")) as f:
        api = f.read()
    a = api.index("void ec_order(")
    body = api[a:api.index("\n}\n", a)]
    assert "std::sort(std::reverse_iterator<std::vector<Rec>::iterator>(recs.begin() + cloud_first[c + 1])" in body
    assert "return a.size < b.size;" in body
