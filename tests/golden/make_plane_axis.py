"""Writes tests/golden/plane_axis.json: the answers of the C++ statement tests/plane_axis_oracle.cpp (pcl::SACSegmentation with SACMODEL_PLANE /
PERPENDICULAR_PLANE / PARALLEL_PLANE, restated from PCL 1.8.1) on the scenes of tests/plane_axis.py.
Run from the repository root: python tests/golden/make_plane_axis.py"""
import json
import math
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import plane_axis as A  # noqa: E402
import plane_axis_oracle as O  # noqa: E402


def main():
    cases = []
    scenes = [("wall", [600, 1200, 300, 3]), ("wall", [900, 300, 200, 5]), ("walls_only", [800, 1])]
    for kind, scene in scenes:
        x = A.wall_zone(*scene) if kind == "wall" else A.walls_only(*scene)
        for model, eps in ((A.PLANE, 0.0), (A.PERP, math.radians(10.0)), (A.PAR, math.radians(10.0)), (A.PERP, 0.05)):
            for optimize in (False, True):
                for order in (0, 1):
                    w = O.plane_ransac_model(x, 0.3, 0.99, 1000, optimize, 12345, order, model, A.Z, eps)
                    cases.append(dict(name="%s%s:m%d:eps%.4f:opt%d:o%d" % (kind, scene, model, eps, optimize, order),
                                      scene_kind=kind, scene=scene, threshold=0.3, probability=0.99, max_iterations=1000,
                                      optimize=optimize, sum_order=order, model=model, axis=list(A.Z), eps_angle=eps,
                                      found=w["found"], iterations=w["iterations"], draws=w["draws"],
                                      best_count=w["best_count"], rejected=w["rejected"],
                                      coeff_bits=w["coeff"].view("uint32").tolist(), n_inliers=len(w["inliers"])))
    with open(os.path.join(HERE, "plane_axis.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_plane_axis.py", "oracle": "tests/plane_axis_oracle.cpp cmo_plane_ransac_model",
                   "cases": cases}, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
