"""Writes tests/golden/ec.json: small clouds of pcl::EuclideanClusterExtraction whose clusters were worked out by hand
(TEST INFRASTRUCTURE ONLY). Each answer below is stated from the geometry, not computed by any implementation; the tests
check that the C++ oracle, the numpy restatement and the GPU all reproduce them."""
import json
import os

import numpy as np

F32 = np.float32
HERE = os.path.dirname(os.path.abspath(__file__))


def row(x, y=0.0, z=0.0, i=0.0):
    return [float(F32(x)), float(F32(y)), float(F32(z)), float(F32(i))]


def r2_ror(t):
    return F32(t * t)                      # the radius outlier removal's (float)(radius * radius)


def r2_ec(t):
    tf = float(F32(t))
    return F32(tf * tf)                    # (float)((double)(float)t * (float)t)


def main():
    cases = []
    # 1. a line: gaps 0.4, 0.4 | 1.2 | 0.3 | 2.7 -> {0,1,2} {3,4} {5}; sizes 3, 2, 1 in seed order, sorted descending
    cases.append(dict(name="line", tolerance=0.5, min_size=1, max_size=2 ** 31 - 1,
                      xyzi=[row(0.0), row(0.4), row(0.8), row(2.0), row(2.3), row(5.0)],
                      clusters=[[0, 1, 2], [3, 4], [5]]))
    # 2. the same line, clusters of 2 .. 2 points only
    cases.append(dict(name="line_min_max", tolerance=0.5, min_size=2, max_size=2,
                      xyzi=cases[0]["xyzi"], clusters=[[3, 4]]))
    # 3. a gap of exactly the tolerance (0.5 is a float: the squared distance equals r2) is not a neighbour: strict <
    cases.append(dict(name="strict_bound", tolerance=0.5, min_size=1, max_size=2 ** 31 - 1,
                      xyzi=[row(0.0), row(0.5), row(1.0)], clusters=[[0], [1], [2]]))
    # 4. indices interleave between two far groups; exact duplicates join their group: {0,2,4,5} and {1,3}, sizes 4, 2
    cases.append(dict(name="interleaved_duplicates", tolerance=0.3, min_size=1, max_size=2 ** 31 - 1,
                      xyzi=[row(0.0), row(10.0), row(0.2), row(10.0), row(0.2), row(0.0)],
                      clusters=[[0, 2, 4, 5], [1, 3]]))
    # 5. a non-float tolerance 0.1: a pair whose float squared distance equals the radius removal's r2 = (float)0.01
    #    lies below the cluster extraction's r2 = (float)((double)0.1f * 0.1f), so the pair is one cluster
    lo, hi = r2_ror(0.1), r2_ec(0.1)
    assert lo < hi
    #    (lo and hi are neighbouring floats and no single-axis step squares to lo: the pair is offset on two axes)
    x, y = F32(0.06755000352859497), F32(0.07373599708080292)
    assert F32(F32(x * x) + F32(y * y)) == lo
    cases.append(dict(name="non_float_tolerance", tolerance=0.1, min_size=1, max_size=2 ** 31 - 1,
                      xyzi=[row(0.0), row(float(x), float(y)), row(3.0)], clusters=[[0, 1], [2]]))
    # 6. a non-finite row belongs to no cluster; the rows around it are 0.2 apart: {0, 2} and {3}
    cases.append(dict(name="non_finite", tolerance=0.25, min_size=1, max_size=2 ** 31 - 1,
                      xyzi=[row(0.0), ["nan", 0.0, 0.0, 0.0], row(0.2), row(4.0)], clusters=[[0, 2], [3]]))
    # 7. min_size > max_size: no cluster
    cases.append(dict(name="min_above_max", tolerance=0.5, min_size=3, max_size=2,
                      xyzi=cases[0]["xyzi"], clusters=[]))
    with open(os.path.join(HERE, "ec.json"), "w") as f:
        json.dump({"cases": cases}, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
