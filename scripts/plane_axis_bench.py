"""SACMODEL_PLANE against SACMODEL_PERPENDICULAR_PLANE (axis z, 10 degrees) in the RANSAC plane search, on one GPU:
the whole 58 k and 233 k-point ROI clouds of scripts/proceed_bench.py, their five ground windows of proceedFront in one
multi-cloud call, and a zone whose wall holds more points than its ground. Per run: wall clock of the blocking call
(median of alternating PLANE / PERPENDICULAR repetitions), the k_plane_score kernel time per call (torch.profiler, in a
pass of its own), iterations, draws and rejected draws, and whether the result equals the C++ statement's
(tests/plane_axis_oracle.cpp). Writes one JSON
document (default profiles/plane_axis_bench.json) with the card's name and power limit."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

from cloud_merger_b200 import ROI_PASSES, CloudMerger, synth
import plane_axis_oracle  # C++ statement of SACSegmentation: the result check beside the timing (bench-side use only)
from oracle import cm_oracle_py as oracle

THR, PROB = float(np.float32(0.3)), float(np.float32(0.99))
PARTS = [(30.0, 30.0, 2.5), (11.0, 19.0, 2.0), (15.0, 4.0, 1.5), (8.0, -4.0, 0.3), (11.0, -15.0, 0.5)]
MODELS = {"PLANE": dict(model=0), "PERPENDICULAR_10deg": dict(model=1, axis=(0.0, 0.0, 1.0), eps_angle=math.radians(10.0))}


def roi_cloud(seed, rings, az):
    c = synth.lidar_cloud(seed, 0, 0, rings, az)
    cur = oracle.transform(c, synth.extrinsic(0, 4)[:3].reshape(-1))
    for (axis, lo, hi, neg) in ROI_PASSES:
        cur = np.ascontiguousarray(cur[oracle.passthrough(cur, axis, lo, hi, bool(neg))])
    return cur


def ground_windows(cloud):
    f32 = np.float32
    zones = [[(0, float(f32(d)), float(f32(f32(d) + f32(l))), 0), (2, float(-f32(z)), float(f32(z)), 0)] for (l, d, z) in PARTS]
    return [np.ascontiguousarray(x) for x, _ in oracle.zone_split(cloud, zones)]


def wall_zone(n_ground=6000, n_wall=12000, n_clutter=3000, seed=0):
    rng = np.random.default_rng(seed)
    g = np.zeros((n_ground, 4), np.float32)
    g[:, 0] = rng.uniform(-6, 6, n_ground); g[:, 1] = rng.uniform(-4, 4, n_ground)
    g[:, 2] = -1.8 + 0.01 * g[:, 0] + rng.uniform(-0.02, 0.02, n_ground)
    w = np.zeros((n_wall, 4), np.float32)
    w[:, 0] = 6.0 + rng.uniform(-0.02, 0.02, n_wall); w[:, 1] = rng.uniform(-4, 4, n_wall); w[:, 2] = rng.uniform(-1.7, 0.3, n_wall)
    c = np.zeros((n_clutter, 4), np.float32)
    c[:, 0] = rng.uniform(-6, 6, n_clutter); c[:, 1] = rng.uniform(-4, 4, n_clutter); c[:, 2] = rng.uniform(-1.5, 0.3, n_clutter)
    x = np.concatenate([g, w, c])
    x[:, 3] = 1.0
    return np.ascontiguousarray(x[rng.permutation(len(x))])


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0]
    except Exception as e:  # the measurement stands without it; say so
        out["power_limit_and_max_sm_clock"] = "not read: %s" % e
    return out


def run_case(label, clouds, steps):
    begin = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    allpts = np.ascontiguousarray(np.concatenate(clouds))
    n = len(allpts)
    cm = CloudMerger(max_sensors=1, max_points_per_sensor=n, max_batch_points=n, max_batch_frames=8)
    buf = cm.upload(allpts)
    call = lambda kw: cm.dev_plane_ransac_multi(buf.ptr, begin, THR, PROB, **kw)
    for kw in MODELS.values():
        for _ in range(3):
            call(kw)
    torch.cuda.synchronize()
    times = {m: [] for m in MODELS}
    res = {}
    for _ in range(steps):   # alternate the two models
        for m, kw in MODELS.items():
            t0 = time.perf_counter()
            res[m] = call(kw)
            times[m].append((time.perf_counter() - t0) * 1e3)
    out = []
    for m, kw in MODELS.items():
        prof_calls = 10
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(prof_calls):
                call(kw)
            torch.cuda.synchronize()
        score_us = sum(e.device_time_total for e in prof.key_averages() if "k_plane_score" in e.key) / prof_calls
        want = [plane_axis_oracle.plane_ransac_model(c, THR, PROB, 1000, True, 12345, 0, **kw) for c in clouds]
        same = all(r["iterations"] == w["iterations"] and r["draws"] == w["draws"] and r["rejected"] == w["rejected"]
                   and r["n_inliers"] == len(w["inliers"]) and r["coeff"].tobytes() == w["coeff"].tobytes()
                   for r, w in zip(res[m], want))
        out.append({"case": label, "model": m, "clouds": len(clouds), "points": n,
                    "wall_ms_median": round(float(np.median(times[m])), 4), "wall_ms_min": round(float(np.min(times[m])), 4),
                    "k_plane_score_us_per_call": round(score_us, 2),
                    "iterations": [r["iterations"] for r in res[m]], "draws": [r["draws"] for r in res[m]],
                    "rejected": [r["rejected"] for r in res[m]], "n_inliers": [r["n_inliers"] for r in res[m]],
                    "normal_z": [round(float(r["coeff"][2]), 4) for r in res[m]], "same_as_cpu_oracle": bool(same)})
    cm.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "plane_axis_bench.json"))
    ap.add_argument("--steps", type=int, default=30)
    a = ap.parse_args()
    runs = []
    for rings, az in ((64, 2048), (128, 4096)):
        roi = roi_cloud(7, rings, az)
        tag = "ROI %dk" % round(len(roi) / 1000)
        runs += run_case(tag + ": whole cloud", [roi], a.steps)
        runs += run_case(tag + ": five ground windows of proceedFront", ground_windows(roi), a.steps)
    runs += run_case("wall-dominated zone (6k ground, 12k wall, 3k clutter)", [wall_zone()], a.steps)
    doc = {"script": "scripts/plane_axis_bench.py", "card": card(), "threshold": THR, "probability": PROB,
           "timing": "wall clock of the blocking dev_plane_ransac_multi call, %d alternating repetitions after 3 warm-up "
                     "calls; k_plane_score: torch.profiler device time over 10 calls" % a.steps, "runs": runs}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
        f.write("\n")
    for r in runs:
        print(json.dumps(r))


if __name__ == "__main__":
    main()
