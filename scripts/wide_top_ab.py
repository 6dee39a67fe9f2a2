#!/usr/bin/env python
"""A/B of the fused-key sort plan: three radix passes sorted frame by frame with a top digit of up to 384 bins (the in-tree
library) against the bit-based plan of four passes.

  wide  the in-tree library as it stands
  base  the in-tree library with CM_NO_WIDE_TOP=1 (the bit-based plan), or --base-lib PATH: another build of the library
        (for instance the parent commit's), selected with CM_LIB_PATH

Each round runs bench.py once per arm on every workload, alternating which arm goes first. Per arm and workload: the
median, min and max of bench's `value`, of the step time and of the sort stage. The first round also dumps the cfg3 and
cfg2 outputs of both arms (bench.py --dump-outputs) and requires them to be bit-identical.

usage: python scripts/wide_top_ab.py [--rounds 5] [--steps 100] [--base-lib PATH] [--out profiles/wide_top_ab.json]"""
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


def gpu_info():
    q = "name,power.limit,clocks.max.sm,driver_version"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    except OSError as e:
        return {"error": str(e)}
    return dict(zip(q.split(","), [s.strip() for s in r.stdout.strip().split(",")])) if r.returncode == 0 else {"error": r.stderr}


def run_bench(env_extra, workload, steps, warmup, dump_dir=None):
    env = dict(os.environ, **env_extra)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", str(steps), "--warmup", str(warmup),
           "--no-e2e", "--no-cpu", "--no-latency"]
    if dump_dir:
        cmd += ["--dump-outputs", dump_dir]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True)
    lines = [s for s in r.stdout.splitlines() if s.startswith("{")]
    if r.returncode != 0 or not lines:
        raise SystemExit("bench.py %s failed (%d):\n%s" % (workload, r.returncode, r.stderr[-3000:]))
    d = json.loads(lines[-1])
    sort = d.get("stages", {}).get("sort", {})
    return {"value": d["value"], "ms_per_step": d["ms_per_step"], "sort_ms": sort.get("ms") if isinstance(sort, dict) else None,
            "stages": d.get("stages"), "launches": d.get("gpu_launches")}


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
    xs = [x for x in xs if x is not None]
    if not xs:
        return None
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs), "all": xs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--workloads", default="cfg3,cfg2,cfg1,cfg5")
    ap.add_argument("--base-lib", default="")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    from cloud_merger_b200 import build as cm_build
    lib = cm_build.build()
    arms = {"wide": {"CM_LIB_PATH": lib},
            "base": {"CM_LIB_PATH": os.path.abspath(a.base_lib)} if a.base_lib else {"CM_LIB_PATH": lib, "CM_NO_WIDE_TOP": "1"}}
    workloads = a.workloads.split(",")
    info = gpu_info()
    print("GPU:", info, flush=True)
    res = {b: {w: [] for w in workloads} for b in arms}
    identical = {}
    with tempfile.TemporaryDirectory() as tmp:
        for rnd in range(a.rounds):
            order = ["base", "wide"] if rnd % 2 == 0 else ["wide", "base"]
            for w in workloads:
                for b in order:
                    dump = os.path.join(tmp, "%s_%s" % (w, b)) if rnd == 0 and w in ("cfg3", "cfg2") else None
                    r = run_bench(arms[b], w, a.steps, a.warmup, dump)
                    res[b][w].append(r)
                    print("round %d %-5s %-5s step %.4f ms  value %.1f  sort %s ms  launches %s" % (
                        rnd, w, b, r["ms_per_step"], r["value"], r["sort_ms"], r["launches"]), flush=True)
                if rnd == 0 and w in ("cfg3", "cfg2"):
                    identical[w] = same_outputs(os.path.join(tmp, w + "_base"), os.path.join(tmp, w + "_wide"))
                    print("%s outputs bit-identical: %s (%s)" % (w, *identical[w]), flush=True)
    summary = {}
    for w in workloads:
        summary[w] = {b: {k: spread([r[k] for r in res[b][w]]) for k in ("value", "ms_per_step", "sort_ms")} for b in arms}
        summary[w]["launches"] = {b: res[b][w][0]["launches"] for b in arms}
        summary[w]["stages_last"] = {b: res[b][w][-1]["stages"] for b in arms}
        s, n = summary[w]["base"]["value"], summary[w]["wide"]["value"]
        summary[w]["wide_vs_base_value"] = n["median"] / s["median"] - 1.0
        summary[w]["ranges_overlap"] = not (n["min"] > s["max"] or s["min"] > n["max"])
        print("%s: value %.1f [%.1f, %.1f] -> %.1f [%.1f, %.1f] (%+.1f %%), ranges overlap: %s" % (
            w, s["median"], s["min"], s["max"], n["median"], n["min"], n["max"], 100 * summary[w]["wide_vs_base_value"],
            summary[w]["ranges_overlap"]), flush=True)
    out = {"gpu": info, "rounds": a.rounds, "steps": a.steps, "base": "library at " + a.base_lib if a.base_lib else "CM_NO_WIDE_TOP=1",
           "identical_outputs": identical, "summary": summary}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
