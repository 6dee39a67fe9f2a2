"""Euclidean cluster extraction on the GPU (cm_dev_euclidean_clusters_multi) next to a one-core CPU run of the C++
statement of PCL's loop (tests/ec_oracle.cpp: seed queue, sorted neighbour lists, std::sort of the clusters), on the clouds
a user clusters after ground removal: one sensor's ROI cloud at two resolutions, its five x-window zone clouds in one call,
a fused 2 M-point cfg3 frame, and a dense blob of 10^5 points in one cell (the worst case of the hook kernel's walk over
its 3 x 3 rows). Tolerance 0.5 m, clusters of 10 .. 25 000 points and of 1 .. INT_MAX points. Reports per case the call
time (host clock around a call and the device output fetch, which ends in a synchronise; median of the repeats), the hook
kernel time (CUDA events, a separate profiled pass), the CPU time, and whether the GPU's clusters equal the oracle's.
Writes one JSON document (default profiles/ec_bench.json) with the GPU's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np

from cloud_merger_b200 import CloudMerger, _lib

import ec_cases as K
import ec_oracle

TOL = 0.5
INT_MAX = 2 ** 31 - 1


def gpu_name_and_power():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers below are still GPU numbers; say what is missing
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ec_bench.json"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cpu-max-points", type=int, default=2_500_000, help="largest case the one-core CPU run is timed on")
    a = ap.parse_args()
    roi58 = K.roi_cloud(7, 64, 2048)
    roi233 = K.roi_cloud(7, 128, 4096)
    cases = [("roi_58k", [roi58]), ("roi_233k", [roi233]), ("zones_5_of_233k", K.zone_clouds(roi233)),
             ("cfg3_fused_2m", [K.fused_frame(3)]), ("dense_blob_100k", [K.dense_blob(5)])]
    res = {"gpu": gpu_name_and_power(), "tolerance": TOL, "reps": a.reps, "cases": []}
    with CloudMerger(max_sensors=1, max_points_per_sensor=1 << 21, max_batch_points=1 << 21, max_batch_frames=16) as cm:
        for name, clouds in cases:
            allpts = np.ascontiguousarray(np.concatenate(clouds))
            begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
            buf = cm.upload(allpts)
            for mn, mx in ((10, 25000), (1, INT_MAX)):
                co = _lib.CmClusterOut()
                cm.set_profiling(False)
                cm.dev_euclidean_clusters_multi(buf.ptr, begin, TOL, mn, mx)  # warm-up of this shape
                cm._check(cm._lib.cm_get_cluster_out(cm._h, co))
                ts = []
                for _ in range(a.reps):
                    t0 = time.perf_counter()
                    cm.dev_euclidean_clusters_multi(buf.ptr, begin, TOL, mn, mx)
                    cm._check(cm._lib.cm_get_cluster_out(cm._h, co))
                    ts.append((time.perf_counter() - t0) * 1e3)
                cm.set_profiling(True)
                cm.dev_euclidean_clusters_multi(buf.ptr, begin, TOL, mn, mx)
                out = cm.euclidean_clusters_out()
                cm.set_profiling(False)
                row = {"case": name, "points": int(len(allpts)), "clouds": len(clouds), "min_size": mn, "max_size": mx,
                       "clusters": int(sum(len(c) for c in out["clusters"])), "unclustered": out["n_unclustered"],
                       "call_ms_median": float(np.median(ts)), "call_ms_min": float(np.min(ts)), "hook_ms": out["hook_ms"],
                       "host_syncs": out["host_syncs"], "launches": int(cm.launch_count())}
                if len(allpts) <= a.cpu_max_points and name != "dense_blob_100k":
                    t0 = time.perf_counter()
                    want = [ec_oracle.euclidean_clusters(c, TOL, mn, mx) for c in clouds]
                    row["cpu_one_core_ms"] = (time.perf_counter() - t0) * 1e3
                    row["clusters_equal"] = all(
                        len(g) == len(w) and all(np.array_equal(gi.astype(np.int64) - begin[c], wi) for gi, wi in zip(g, w))
                        for c, (g, w) in enumerate(zip(out["clusters"], want)))
                else:
                    # PCL's loop sorts a neighbour list of ~10^5 entries for each of the 10^5 points: not run
                    row["cpu_one_core_ms"] = None
                res["cases"].append(row)
                print(json.dumps(row), flush=True)
            buf.free()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")
    print(json.dumps({"gpu": res["gpu"]}))


if __name__ == "__main__":
    main()
