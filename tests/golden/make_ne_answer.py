"""Writes tests/golden/ne.json: small normal estimation cases and the bits of their answers (nx ny nz curvature per
point) under the shared trig rule. Every answer is worked out twice and must agree bit for bit: by the C++ statement
(tests/ne_oracle.cpp, cm_ne_math.h) and step by step by the numpy restatement of PCL's source (tests/ne_np.py). The plane
cases are also derived by hand in tests/test_ne_oracle.py. Run from tests/: python golden/make_ne_answer.py"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import ne_cases as K  # noqa: E402
import ne_np as NP  # noqa: E402
import ne_oracle as O  # noqa: E402

F32 = np.float32


def main():
    tri = K.cloud([[0, 0, 0], [0.1, 0, 0], [0, 0.1, 0]])                    # a plane z = 0: normal (0, 0, +-1), curvature 0
    tet = K.cloud([[0, 0, 0], [0.1, 0, 0], [0, 0.1, 0], [0, 0, 0.05]])      # the closed form
    cases = [
        ("three_points_plane", tri, 0.5, (0, 0, 1)),
        ("three_points_plane_flipped", tri, 0.5, (0, 0, -1)),
        ("tetrahedron", tet, 0.5, (0, 0, 0)),
        ("two_points_nan", K.cloud([[0, 0, 0], [0.1, 0, 0]]), 0.5, (0, 0, 0)),
        ("duplicates", K.cloud([[1, 2, 3]] * 3), 0.5, (0, 0, 0)),
        ("small_groups", K.small_groups(0.3), 0.3, (0, 0, 0)),
        ("lattice_ties", K.lattice(3, 0.25), 0.3, (1, 1, 1)),
        ("eigen_family", K.eigen_family(5, 0.3)[:200], 0.3, (0.5, -0.5, 2.0)),
    ]
    out = {"about": "pcl::NormalEstimation (PCL 1.8.1) radius search, shared trig rule: bits of nx ny nz curvature",
           "cases": []}
    for name, c, r, vp in cases:
        got = O.normals(c, r, vp)
        steps = NP.normals(c, r, vp)
        assert np.array_equal(got.view(np.uint32), steps.view(np.uint32)), name
        out["cases"].append({"name": name, "radius": r, "viewpoint": [float(v) for v in vp],
                             "xyzi": [float(v) for v in np.asarray(c, F32).reshape(-1)],
                             "bits": np.ascontiguousarray(got, F32).view(np.uint32).tolist()})
    with open(os.path.join(HERE, "ne.json"), "w") as f:
        json.dump(out, f, indent=0)


if __name__ == "__main__":
    main()
