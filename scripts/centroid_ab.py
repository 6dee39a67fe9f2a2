#!/usr/bin/env python
"""A/B of k_voxel_centroid's point gather, both builds in one process tree on one GPU.

  async  the in-tree library: the count sweep of the next tile issues its point gathers as cp.async (CE_ASYNC_GATHER 1)
  sync   the same sources with -DCE_ASYNC_GATHER=0 (variants/libcm_ce_sync.so, selected with CM_LIB_PATH): the tile's item
         phase reads its records again and gathers its points with synchronous loads

Each round runs bench.py once per build on cfg3 (the flagship batch), cfg5 (leaf sweep; its 0.05 m leaf is reported) and
cfg2, alternating which build goes first. Per build and workload: the median of the step time, of bench's `value` and of
the centroid stage time, with their min and max. The first round also dumps the cfg3 and cfg2 outputs of both builds
(bench.py --dump-outputs) and requires them to be bit-identical.

usage: python scripts/centroid_ab.py [--rounds 5] [--steps 100] [--out profiles/centroid_ab.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = ("cfg3", "cfg5", "cfg2")
CFG5_LEAF = "leaf_0.05"


def build_both():
    from cloud_merger_b200 import build as cm_build
    lib_async = cm_build.build()
    env = dict(os.environ, PATH=os.path.dirname(cm_build._nvcc()) + os.pathsep + os.environ.get("PATH", ""))  # the script calls `nvcc`
    out = subprocess.run(["bash", os.path.join(ROOT, "scripts", "build_variant.sh"), "ce_sync", "-DCE_ASYNC_GATHER=0", "cm_voxel.cu"],
                         check=True, capture_output=True, text=True, env=env).stdout
    lib_sync = out.strip().splitlines()[-1]
    return {"async": lib_async, "sync": lib_sync}


def gpu_info():
    q = "name,power.limit,clocks.max.sm,driver_version"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    except OSError as e:
        return {"error": str(e)}
    return dict(zip(q.split(","), [s.strip() for s in r.stdout.strip().split(",")])) if r.returncode == 0 else {"error": r.stderr}


def run_bench(lib, workload, steps, warmup, dump_dir=None):
    env = dict(os.environ, CM_LIB_PATH=lib)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", str(steps), "--warmup", str(warmup),
           "--no-e2e", "--no-cpu", "--no-latency"]
    if dump_dir:
        cmd += ["--dump-outputs", dump_dir]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True)
    lines = [s for s in r.stdout.splitlines() if s.startswith("{")]
    if r.returncode != 0 or not lines:
        raise SystemExit("bench.py %s failed (%d):\n%s" % (workload, r.returncode, r.stderr[-3000:]))
    d = json.loads(lines[-1])
    st = d["stages"]
    cent = st[CFG5_LEAF]["centroid_ms"] if workload == "cfg5" else st["centroid"]["ms"]
    return {"value": d["value"], "ms_per_step": d["ms_per_step"], "centroid_ms": cent}


def same_outputs(dir_a, dir_b):
    names = sorted(f for f in os.listdir(dir_a) if f.endswith(".npy"))
    if not names or names != sorted(f for f in os.listdir(dir_b) if f.endswith(".npy")):
        return False, "different file sets"
    for f in names:
        a, b = np.load(os.path.join(dir_a, f)), np.load(os.path.join(dir_b, f))
        if a.shape != b.shape or a.dtype != b.dtype or a.tobytes() != b.tobytes():
            return False, f
    return True, "%d arrays" % len(names)


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs), "all": xs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    libs = build_both()
    info = gpu_info()
    print("GPU:", info, flush=True)
    res = {b: {w: [] for w in WORKLOADS} for b in libs}
    identical = {}
    with tempfile.TemporaryDirectory() as tmp:
        for rnd in range(a.rounds):
            order = ["sync", "async"] if rnd % 2 == 0 else ["async", "sync"]
            for w in WORKLOADS:
                for b in order:
                    dump = os.path.join(tmp, "%s_%s" % (w, b)) if rnd == 0 and w != "cfg5" else None
                    r = run_bench(libs[b], w, a.steps, a.warmup, dump)
                    res[b][w].append(r)
                    print("round %d %-5s %-5s step %.4f ms  value %.1f  centroid %.4f ms" % (rnd, w, b, r["ms_per_step"], r["value"],
                                                                                        r["centroid_ms"]), flush=True)
                if rnd == 0 and w != "cfg5":
                    identical[w] = same_outputs(os.path.join(tmp, w + "_sync"), os.path.join(tmp, w + "_async"))
                    print("%s outputs bit-identical: %s (%s)" % (w, *identical[w]), flush=True)
    summary = {}
    for w in WORKLOADS:
        summary[w] = {}
        for b in libs:
            summary[w][b] = {k: spread([r[k] for r in res[b][w]]) for k in ("ms_per_step", "value", "centroid_ms")}
        s, n = summary[w]["sync"], summary[w]["async"]
        summary[w]["async_vs_sync"] = {
            "value": n["value"]["median"] / s["value"]["median"] - 1.0,
            "ms_per_step": n["ms_per_step"]["median"] / s["ms_per_step"]["median"] - 1.0,
            "centroid_ms": n["centroid_ms"]["median"] / s["centroid_ms"]["median"] - 1.0}
        print("%s%s: centroid %.4f [%.4f, %.4f] -> %.4f [%.4f, %.4f] ms (%+.1f %%); step %.4f [%.4f, %.4f] -> %.4f [%.4f, %.4f] ms; "
              "value %+.1f %%" % (w, " " + CFG5_LEAF if w == "cfg5" else "",
                                  s["centroid_ms"]["median"], s["centroid_ms"]["min"], s["centroid_ms"]["max"],
                                  n["centroid_ms"]["median"], n["centroid_ms"]["min"], n["centroid_ms"]["max"],
                                  100 * summary[w]["async_vs_sync"]["centroid_ms"],
                                  s["ms_per_step"]["median"], s["ms_per_step"]["min"], s["ms_per_step"]["max"],
                                  n["ms_per_step"]["median"], n["ms_per_step"]["min"], n["ms_per_step"]["max"],
                                  100 * summary[w]["async_vs_sync"]["value"]), flush=True)
    out = {"gpu": info, "rounds": a.rounds, "steps": a.steps, "warmup": a.warmup,
           "what": "bench.py --no-e2e --no-cpu --no-latency per build and workload, alternating; centroid = stage time of the "
                   "last timed step (cfg5: its %s leaf); step = whole step (cfg5: all seven leaves)" % CFG5_LEAF,
           "outputs_bit_identical": {w: v[0] for w, v in identical.items()}, "summary": summary}
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    return 0 if all(v[0] for v in identical.values()) else 1


if __name__ == "__main__":
    sys.exit(main())
