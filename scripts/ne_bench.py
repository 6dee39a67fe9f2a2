"""Normal estimation on the GPU (cm_dev_normals_multi) next to a one-core CPU run of the C++ statement of PCL's loop
(tests/ne_oracle.cpp: sorted neighbour lists, the nine running sums, pcl::eigen33 through cm_ne_math.h), on the clouds a
user estimates normals on: one sensor's ROI cloud at two resolutions, its five x-window zone clouds in one call, a fused
2.1 M-point cfg3 frame, and a dense blob of 10^5 points within one radius (every query sees the whole cloud: the CTA
kernel's multi-walk path). Radii 0.1 / 0.3 / 0.5 m. Reports per case the call time (host clock around a call and
cm_get_normal_out, which ends in a synchronise; median of the repeats), the warp and CTA kernel times (CUDA events, a
separate profiled pass), the queries per path, the CPU time on one core and whether the GPU's bits equal the statement's
(both except for the blob and the 2 M frame). Writes one JSON document (default profiles/ne_bench.json) with the GPU's
name and power limit."""
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

import ne_cases as K
import ne_oracle

RADII = (0.1, 0.3, 0.5)


def gpu_name_and_power():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers below are still GPU numbers; say what is missing
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ne_bench.json"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--no-cpu", action="store_true", help="skip the one-core CPU runs")
    a = ap.parse_args()
    roi58 = K.roi_cloud(7, 64, 2048)
    roi233 = K.roi_cloud(7, 128, 4096)
    cases = [("roi_58k", [roi58]), ("roi_233k", [roi233]), ("zones_5_of_233k", K.zone_clouds(roi233)),
             ("cfg3_fused_2m", [K.fused_frame(3)]), ("dense_blob_100k", [K.dense_blob(5, 100000, 0.1)])]
    res = {"gpu": gpu_name_and_power(), "radii": list(RADII), "reps": a.reps, "cases": []}
    with CloudMerger(max_sensors=1, max_points_per_sensor=1 << 21, max_batch_points=1 << 22, max_batch_frames=16) as cm:
        for name, clouds in cases:
            allpts = np.ascontiguousarray(np.concatenate(clouds))
            begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
            buf = cm.upload(allpts)
            radii = (0.1,) if name == "dense_blob_100k" else RADII  # the blob is built for one radius
            for r in radii:
                no = _lib.CmNormalOut()
                cm.set_profiling(False)
                cm.dev_normals_multi(buf.ptr, begin, r)  # warm-up of this shape
                cm._check(cm._lib.cm_get_normal_out(cm._h, no))
                reps = a.reps if name != "dense_blob_100k" else 2
                ts = []
                for _ in range(reps):
                    t0 = time.perf_counter()
                    cm.dev_normals_multi(buf.ptr, begin, r)
                    cm._check(cm._lib.cm_get_normal_out(cm._h, no))
                    ts.append((time.perf_counter() - t0) * 1e3)
                cm.set_profiling(True)
                cm.dev_normals_multi(buf.ptr, begin, r)
                out = cm.normals_out()
                cm.set_profiling(False)
                row = {"case": name, "points": int(len(allpts)), "clouds": len(clouds), "radius": r,
                       "call_ms_median": float(np.median(ts)), "call_ms_min": float(np.min(ts)),
                       "warp_ms": out["warp_ms"], "cta_ms": out["cta_ms"], "max_neighbors": out["max_neighbors"],
                       "n_warp": out["n_warp"], "n_cta": out["n_cta"], "n_multi": out["n_multi"],
                       "nan": int(sum(out["n_nan"])), "host_syncs": out["host_syncs"], "launches": int(cm.launch_count())}
                if not a.no_cpu and name not in ("dense_blob_100k", "cfg3_fused_2m"):
                    ne_oracle.set_threads(1)
                    t0 = time.perf_counter()
                    want = [ne_oracle.normals(c, r) for c in clouds]
                    row["cpu_one_core_ms"] = (time.perf_counter() - t0) * 1e3
                    ne_oracle.set_threads(0)
                    got = out["normals"]
                    row["bits_equal"] = all(np.array_equal(got[begin[c]:begin[c + 1]].view(np.uint32), w.view(np.uint32))
                                            for c, w in enumerate(want))
                else:
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
