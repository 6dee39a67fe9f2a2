"""Writes tests/golden/sor.json: known answers of pcl::StatisticalOutlierRemoval (PCL 1.8.1 applyFilterIndices) on clouds
small enough to check by hand -- no oracle code is imported. Every step is written out below with plain Python doubles and
explicit float32 rounding (numpy scalars). Coordinates are stored as the hex bits of their float32 values, so NaN and
+-inf survive the trip.

Cases (x, y, z; intensity 0):
  line          x = 0, 1, 2, 3, 10 on a line, mean_k 2: distances 1.5, 1, 1, 1.5, 7.5 (the roots are exact), mean 2.5,
                variance (62.75 - 12.5^2 / 5) / 4 = 7.875, threshold 2.5 + 2.80624... -> the point at 10 is removed;
  line_negative the same with negative: only the point at 10 is kept;
  nan_rows      the line with a NaN, an inf and a -inf row between its points: those get distance 0, are not valid,
                and are kept (0 <= threshold);
  roots         points at squared distances 2 and 3 from their neighbours (inexact roots), both sqrt modes, std_mul 0;
  too_few       two finite points and a NaN row with mean_k 2: every point is kept, distances 0.

Run: python tests/golden/make_sor_answer.py
"""
import json
import math
import os

import numpy as np

F = np.float32
HERE = os.path.dirname(os.path.abspath(__file__))


def f32(v):
    return F(v)


def sq_dist(a, b):
    """FLANN L2_Simple in float32: (dx*dx + dy*dy) + dz*dz, each operation rounded."""
    dx, dy, dz = f32(a[0] - b[0]), f32(a[1] - b[1]), f32(a[2] - b[2])
    return f32(f32(f32(dx * dx) + f32(dy * dy)) + f32(dz * dz))


def answer(pts, mean_k, std_mul, negative, sqrt_mode):
    finite = [i for i, p in enumerate(pts) if all(math.isfinite(float(v)) for v in p[:3])]
    valid = len(finite)
    too_few = 0 < valid <= mean_k
    dist = [F(0.0)] * len(pts)
    if valid and not too_few:
        for i in finite:
            d = sorted(sq_dist(pts[i], pts[j]) for j in finite)[: mean_k + 1]
            s = 0.0
            for k in range(1, mean_k + 1):
                s += float(np.sqrt(d[k])) if sqrt_mode == 0 else math.sqrt(float(d[k]))
            dist[i] = f32(s / mean_k)
    total = 0.0
    sq_total = 0.0
    for v in dist:
        total += float(v)
        sq_total += float(f32(v * v))
    mean = total / valid if valid else math.nan
    variance = (sq_total - total * total / valid) / (valid - 1) if valid > 1 else math.nan
    stddev = math.sqrt(variance) if variance >= 0 else math.nan
    threshold = mean + std_mul * stddev
    kept = []
    for i, v in enumerate(dist):
        removed = (float(v) <= threshold) if negative else (float(v) > threshold)
        if too_few or not removed:
            kept.append(i)
    return dist, kept, mean, stddev, threshold, valid, too_few


def hexf(v):
    return "%08x" % int(np.array([v], F).view(np.uint32)[0])


def hexd(v):
    return "%016x" % int(np.array([v], np.float64).view(np.uint64)[0])


def main():
    line = [[0, 0, 0], [1, 0, 0], [2, 0, 0], [3, 0, 0], [10, 0, 0]]
    nan_rows = [line[0], [np.nan, 0, 0], line[1], line[2], [0, np.inf, 0], line[3], [0, 0, -np.inf], line[4]]
    roots = [[0, 0, 0], [1, 1, 0], [2, 2, 0], [3, 2, 1], [4, 3, 2], [9, 9, 9]]
    cases = [("line", line, 2, 1.0, 0, 0), ("line_negative", line, 2, 1.0, 1, 0), ("nan_rows", nan_rows, 2, 1.0, 0, 0),
             ("roots_float_sqrt", roots, 2, 0.0, 0, 0), ("roots_double_sqrt", roots, 2, 0.0, 0, 1),
             ("too_few", [[0, 0, 0], [1, 0, 0], [np.nan, 0, 0]], 2, 1.0, 0, 0)]
    out = []
    for name, rows, mean_k, std_mul, negative, sqrt_mode in cases:
        pts = [[F(v) for v in r] + [F(0)] for r in rows]
        dist, kept, mean, stddev, thr, valid, too_few = answer(pts, mean_k, std_mul, negative, sqrt_mode)
        out.append({"name": name, "xyzi": [[hexf(v) for v in p] for p in pts], "mean_k": mean_k, "std_mul": std_mul,
                    "negative": negative, "sqrt_mode": sqrt_mode, "distances": [hexf(v) for v in dist], "kept": kept,
                    "mean": hexd(mean), "stddev": hexd(stddev), "threshold": hexd(thr), "n_valid": valid,
                    "too_few": too_few})
    with open(os.path.join(HERE, "sor.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
