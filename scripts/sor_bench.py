"""Statistical outlier removal on the GPU (cm_dev_statistical_outlier_multi) next to the numpy / scipy restatement of
tests/sor_np.py on one core (a cKDTree search, as PCL's FLANN tree, plus PCL's loops), on the clouds a user of the
preprocessing chain filters: one sensor's ROI cloud at two resolutions, its five x-window zone clouds in one call, and a
fused 2 M-point cfg3 frame; mean_k 10, 50 and 127, std_mul 1. Reports per case the call time (host clock around a call
that ends in a device synchronise, median of the repeats), the kNN and sums kernel times (CUDA events, a separate
profiled pass), the sum path every cloud took, the CPU time, and whether the GPU result equals the restatement bit for
bit. Writes one JSON document (default profiles/sor_bench.json) with the GPU's name and power limit."""
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

from cloud_merger_b200 import CloudMerger

import sor_cases as K
import sor_np


def gpu_name_and_power():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers below are still GPU numbers; say what is missing
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sor_bench.json"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cpu-max-points", type=int, default=300000, help="largest case the one-core CPU run is timed on")
    a = ap.parse_args()
    roi58 = K.roi_cloud(7, 64, 2048)
    roi233 = K.roi_cloud(7, 128, 4096)
    cases = [("roi_58k", [roi58]), ("roi_233k", [roi233]), ("zones_5_of_233k", K.zone_clouds(roi233)),
             ("cfg3_fused_2m", [K.fused_frame(3)])]
    res = {"gpu": gpu_name_and_power(), "std_mul": 1.0, "reps": a.reps, "cases": []}
    with CloudMerger(max_sensors=1, max_points_per_sensor=1 << 21, max_batch_points=1 << 21, max_batch_frames=16) as cm:
        for name, clouds in cases:
            allpts = np.ascontiguousarray(np.concatenate(clouds))
            begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
            buf = cm.upload(allpts)
            for mean_k in (10, 50, 127):
                cm.set_profiling(False)
                cm.dev_statistical_outlier_multi(buf.ptr, begin, mean_k, 1.0)  # warm-up of this shape
                cm.statistical_outlier_out()
                ts = []
                for _ in range(a.reps):
                    t0 = time.perf_counter()
                    cm.dev_statistical_outlier_multi(buf.ptr, begin, mean_k, 1.0)
                    cm.zone_out_raw()
                    ts.append((time.perf_counter() - t0) * 1e3)
                cm.set_profiling(True)
                cm.dev_statistical_outlier_multi(buf.ptr, begin, mean_k, 1.0)
                out = cm.statistical_outlier_out()
                cm.set_profiling(False)
                row = {"case": name, "points": int(len(allpts)), "clouds": len(clouds), "mean_k": mean_k,
                       "call_ms_median": float(np.median(ts)), "call_ms_min": float(np.min(ts)),
                       "knn_ms": out["knn_ms"], "sums_ms": out["sums_ms"],
                       "sum_path": [c["sum_path"] for c in out["clouds"]],
                       "kept": cm.zone_out_raw()[2][-1]}
                if len(allpts) <= a.cpu_max_points or mean_k == 10:
                    t0 = time.perf_counter()
                    want = [sor_np.sor_cloud(c, mean_k, 1.0, workers=1 if len(allpts) <= a.cpu_max_points else -1)
                            for c in clouds]
                    cpu = (time.perf_counter() - t0) * 1e3
                    row["cpu_one_core_ms"] = cpu if len(allpts) <= a.cpu_max_points else None
                    d = np.concatenate([w["distances"] for w in want])
                    row["distances_bit_equal"] = bool(np.array_equal(d.view(np.uint32), out["distances"].view(np.uint32)))
                    zones = cm.zone_out()
                    row["survivors_equal"] = all(
                        np.array_equal(zi.astype(np.int64) - begin[c], np.nonzero(w["keep"])[0])
                        for c, ((_, zi), w) in enumerate(zip(zones, want)))
                else:
                    row["cpu_one_core_ms"] = None
                res["cases"].append(row)
                print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")
    print(json.dumps({"gpu": res["gpu"]}))


if __name__ == "__main__":
    main()
