"""Cost of pcl::CropBox stages in K1 (cm_set_crop_boxes) on BASELINE config 3: a device-resident batch of F frames x 8
sensors x 256k points through cm_run_batch, with 0, 1 (the ego box: negative, translated and yawed), 2 and 8 boxes. The arms
alternate round by round on the same handle and inputs. Per arm: the transform_crop stage time (CUDA events, cm_stage_ms)
and the whole step time (CUDA events around --steps back-to-back steps), median and spread over the rounds. Writes JSON
(with the card's name and power limit) to profiles/ or --out and prints it.

    python scripts/crop_box_bench.py [--frames 16] [--steps 20] [--rounds 5] [--out profiles/crop_box_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import crop_box_cases as K
from cloud_merger_b200 import CloudMerger, make_layout, synth

ARMS = {
    0: [],
    1: [K.EGO],
    2: [K.EGO, K.box((-0.5, -0.75, 1.5), (1.5, 0.75, 2.25), negative=True)],   # + a roof rack
    8: [K.EGO] + [K.box((-6.0 + 1.5 * k, 2.0, -0.5), (-5.0 + 1.5 * k, 2.5, 0.5), rotation=(0.0, 0.0, 0.1 * k), negative=True)
                  for k in range(7)],
}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0]
        name, power, clock = [v.strip() for v in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers without the card are still reported, marked as such
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "crop_box_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("crop_box_bench.py: no CUDA device")
    spec = synth.CONFIGS["cfg3"]
    S, n, F = spec["sensors"], spec["rings"] * spec["azimuth"], a.frames
    host = np.empty((F * S, n, 4), np.float32)
    for f in range(F):
        for s in range(S):
            host[f * S + s] = synth.lidar_cloud(3000, s, f, spec["rings"], spec["azimuth"])
    dev = torch.from_numpy(host.reshape(-1).view(np.uint8)).cuda()
    cm = CloudMerger(max_sensors=S, max_points_per_sensor=n, max_point_step=16, max_batch_points=F * S * n,
                     max_batch_frames=F)
    for s in range(S):
        cm.set_extrinsic(s, synth.extrinsic(s, S))
    cm.set_crop(spec["passes"])
    cm.set_voxel(spec["leaf"], spec["min_points"], True)
    segs = cm.make_segments([(dev.data_ptr() + (f * S + s) * n * 16, n, make_layout(), s, f) for f in range(F) for s in range(S)])
    stream = torch.cuda.current_stream().cuda_stream
    res = {k: {"k1_ms": [], "step_ms": [], "survivors": None, "key_bytes": None} for k in ARMS}
    for arm, boxes in ARMS.items():   # warm every arm
        cm.set_crop_boxes([K.to_cm(b) for b in boxes])
        for _ in range(3):
            cm.run_batch(segs, stream=stream)
        cm.sync()
    for _ in range(a.rounds):
        for arm, boxes in ARMS.items():
            cm.set_crop_boxes([K.to_cm(b) for b in boxes])
            cm.set_profiling(True)
            cm.run_batch(segs, stream=stream)
            cm.sync()
            res[arm]["k1_ms"].append(cm.stage_ms("transform_crop"))
            cm.set_profiling(False)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                cm.run_batch(segs, stream=stream)
            e1.record()
            cm.sync()
            res[arm]["step_ms"].append(e0.elapsed_time(e1) / a.steps)
            st = cm.stats()
            assert st.device_error == 0
            res[arm]["survivors"] = int(st.survivors)
            res[arm]["key_bytes"] = int(st.key_bytes)
    base_k1 = float(np.median(res[0]["k1_ms"]))
    out = {"what": "cfg3 batch, cm_run_batch, CropBox stages after the ROI box", "card": card(), "frames": F,
           "points_per_step": F * S * n, "steps_per_round": a.steps, "rounds": a.rounds, "arms": {}}
    for arm, r in res.items():
        k1, step = np.asarray(r["k1_ms"]), np.asarray(r["step_ms"])
        out["arms"][str(arm)] = {
            "boxes": arm, "k1_ms_median": float(np.median(k1)), "k1_ms_min": float(k1.min()), "k1_ms_max": float(k1.max()),
            "step_ms_median": float(np.median(step)), "step_ms_min": float(step.min()), "step_ms_max": float(step.max()),
            "k1_vs_no_box": float(np.median(k1)) / base_k1, "survivors": r["survivors"], "key_bytes": r["key_bytes"],
            "mpoints_per_s": F * S * n / (float(np.median(step)) / 1e3) / 1e6}
    cm.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
