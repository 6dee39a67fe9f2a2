#!/usr/bin/env python
"""A/B of two builds of the library on the four filters that search the sorted cell keys: the radius outlier removal, the
statistical outlier removal, the Euclidean cluster extraction and the normal estimation.

  new   the in-tree library
  base  another build of the same C ABI (for instance the parent commit's), given with --base-lib

Every round runs one process per build (CM_LIB_PATH selects the library), alternating which build goes first. A process
runs the cases of scripts/outlier_bench.py, sor_bench.py, ec_bench.py and ne_bench.py on the same seeded inputs, each
with the cell table and with the binary searches (CM_ROR_NO_TABLE / CM_SOR_NO_TABLE / CM_EC_NO_TABLE / CM_NE_NO_TABLE),
and times every call on the host clock up to the output's stream synchronise. The outputs of both builds are compared bit
for bit in every round. Per case and build: the median over the rounds of the per-round median call time, and the spread
(max - min) of those per-round medians. The normal estimation's dense 10^5-point blob (16 s a call, k_ne_cta's multi-walk
path) is left out.

usage: python scripts/cell_search_ab.py --base-lib <path> [--rounds 3] [--seconds 1.0] [--filters ror,sor,ec,ne] [--out <json>]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np

NO_TABLE = {"ror": "CM_ROR_NO_TABLE", "sor": "CM_SOR_NO_TABLE", "ec": "CM_EC_NO_TABLE", "ne": "CM_NE_NO_TABLE"}


def make_inputs(path):
    """The clouds of the four benchmarks, by name, into one .npz (cloud name -> [n, 4] float32, plus its cloud offsets)."""
    from cloud_merger_b200 import ROI_PASSES, synth
    import sor_cases as K
    arrays = {}

    def put(name, clouds):
        arrays[name] = np.ascontiguousarray(np.concatenate(clouds))
        arrays[name + ":begin"] = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)

    for frames in (1, 16):  # outlier_bench.py
        S, rings, az = 4, 128, 1024
        clouds = []
        for f in range(frames):
            for s in range(S):
                c = synth.lidar_cloud(2000, s, f, rings, az)
                m = synth.extrinsic(s, S)[:3]
                xyz = (c[:, :3].astype(np.float64) @ m[:, :3].T.astype(np.float64) + m[:, 3]).astype(np.float32)
                keep = np.ones(len(c), bool)
                for axis, lo, hi, _ in ROI_PASSES:
                    keep &= (xyz[:, axis] >= lo) & (xyz[:, axis] <= hi)
                clouds.append(np.column_stack([xyz[keep], c[keep, 3]]).astype(np.float32))
        put("ror_frames_%d" % frames, [np.concatenate(clouds)])
    roi233 = K.roi_cloud(7, 128, 4096)
    put("roi_58k", [K.roi_cloud(7, 64, 2048)])
    put("roi_233k", [roi233])
    put("zones_5_of_233k", K.zone_clouds(roi233))
    put("cfg3_fused_2m", [K.fused_frame(3)])
    import ec_cases
    put("ec_dense_blob_100k", [ec_cases.dense_blob(5)])
    np.savez(path, **arrays)


def cases(filters):
    """(filter, cloud name, parameters) of every timed case of the given filters."""
    out = [("ror", "ror_frames_%d" % f, {"radius": float(np.float32(0.15)), "min_neighbors": 1}) for f in (1, 16)]
    big = ("roi_58k", "roi_233k", "zones_5_of_233k", "cfg3_fused_2m")
    out += [("sor", c, {"mean_k": k}) for c in big for k in (10, 50, 127)]
    out += [("ec", c, {"min_size": mn, "max_size": mx}) for c in big + ("ec_dense_blob_100k",)
            for mn, mx in ((10, 25000), (1, 2 ** 31 - 1))]
    out += [("ne", c, {"radius": r}) for c in big for r in (0.1, 0.3, 0.5)]
    return [c for c in out if c[0] in filters]


def child(inputs, seconds, filters, dump):
    """One build: every case in both table modes; prints {case id: [call ms]} and writes the outputs to `dump`."""
    from cloud_merger_b200 import CloudMerger, _lib
    data = np.load(inputs)
    times, outs = {}, {}
    with CloudMerger(max_sensors=1, max_points_per_sensor=1 << 22, max_batch_points=1 << 22, max_batch_frames=16) as cm:
        bufs = {}
        for filt, name, prm in cases(filters):
            pts, begin = data[name], data[name + ":begin"]
            if name not in bufs:
                bufs.clear()
                bufs[name] = cm.upload(pts)
            buf = bufs[name]
            if filt == "ror":
                def call():
                    cm.dev_radius_outlier_multi(buf.ptr, begin, prm["radius"], prm["min_neighbors"])
                    cm._check(cm._lib.cm_get_zone_out(cm._h, _lib.CmZoneOut()))
            elif filt == "sor":
                def call():
                    cm.dev_statistical_outlier_multi(buf.ptr, begin, prm["mean_k"], 1.0)
                    cm._check(cm._lib.cm_get_zone_out(cm._h, _lib.CmZoneOut()))
            elif filt == "ec":
                def call():
                    cm.dev_euclidean_clusters_multi(buf.ptr, begin, 0.5, prm["min_size"], prm["max_size"])
                    cm._check(cm._lib.cm_get_cluster_out(cm._h, _lib.CmClusterOut()))
            else:
                def call():
                    cm.dev_normals_multi(buf.ptr, begin, prm["radius"])
                    cm._check(cm._lib.cm_get_normal_out(cm._h, _lib.CmNormalOut()))
            for mode in ("table", "no_table"):
                if mode == "no_table":
                    os.environ[NO_TABLE[filt]] = "1"
                else:
                    os.environ.pop(NO_TABLE[filt], None)
                key = "%s|%s|%s|%s" % (filt, name, ",".join("%s=%s" % kv for kv in sorted(prm.items())), mode)
                t0 = time.perf_counter()
                call()  # warm-up of this shape
                first = time.perf_counter() - t0
                reps = int(min(20, max(3, seconds / max(first, 1e-6))))
                ts = []
                for _ in range(reps):
                    t0 = time.perf_counter()
                    call()
                    ts.append((time.perf_counter() - t0) * 1e3)
                times[key] = ts
                if filt in ("ror", "sor"):
                    zones = cm.zone_out()
                    outs[key + "|idx"] = np.concatenate([z[1] for z in zones])
                    outs[key + "|zones"] = np.array([len(z[1]) for z in zones], np.int64)
                    if filt == "sor":
                        outs[key + "|dist"] = cm.statistical_outlier_out()["distances"].view(np.uint32)
                elif filt == "ec":
                    o = cm.euclidean_clusters_out()
                    outs[key + "|begin"] = o["begin"]
                    outs[key + "|idx"] = np.concatenate([np.concatenate(c) if c else np.zeros(0, np.uint32)
                                                         for c in o["clusters"]])
                else:
                    outs[key + "|normals"] = cm.normals_out()["normals"].view(np.uint32)
            os.environ.pop(NO_TABLE[filt], None)
    np.savez(dump, **outs)
    print(json.dumps(times))


def summarize(res, per, out):
    """Per case and build: the median and the spread of the per-round medians; written to `out` (after every round, so an
    interrupted run keeps the rounds it finished)."""
    worst = 0.0
    for k, v in per.items():
        row = {}
        for b, meds in v.items():
            row[b] = {"median_ms": float(np.median(meds)), "spread_ms": float(np.max(meds) - np.min(meds)),
                      "round_medians_ms": meds}
        row["new_minus_base_ms"] = row["new"]["median_ms"] - row["base"]["median_ms"]
        noise = max(row["new"]["spread_ms"], row["base"]["spread_ms"])
        row["slower_than_spread"] = row["new_minus_base_ms"] > noise
        res["cases"][k] = row
        worst = max(worst, row["new_minus_base_ms"] / row["base"]["median_ms"])
    res["bit_identical"] = not res["mismatches"]
    res["n_slower_than_spread"] = sum(r["slower_than_spread"] for r in res["cases"].values())
    res["worst_relative_change"] = worst
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    return worst


def gpu_name_and_power():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers below are still GPU numbers; say what is missing
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-lib", help="the other build (required unless --child)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0, help="timed calls per case: about this long, 3 .. 20 calls")
    ap.add_argument("--filters", default="ror,sor,ec,ne", help="comma-separated subset of ror, sor, ec, ne")
    ap.add_argument("--out", default=None, help="JSON result (default: a temporary directory)")
    ap.add_argument("--child", nargs=2, metavar=("INPUTS", "DUMP"), help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        return child(a.child[0], a.seconds, a.filters.split(","), a.child[1])
    if not a.base_lib:
        ap.error("--base-lib is required")
    from cloud_merger_b200 import build as cm_build
    libs = {"new": cm_build.LIB, "base": os.path.abspath(a.base_lib)}
    tmp = tempfile.mkdtemp(prefix="cell_search_ab_")
    out = a.out or os.path.join(tmp, "cell_search_ab.json")
    inputs = os.path.join(tmp, "inputs.npz")
    make_inputs(inputs)
    res = {"gpu": gpu_name_and_power(), "libs": {b: os.path.relpath(v, ROOT) for b, v in libs.items()}, "rounds": a.rounds,
           "seconds": a.seconds, "mismatches": [], "cases": {}}
    per = {}  # case -> build -> per-round medians
    for r in range(a.rounds):
        order = ("new", "base") if r % 2 == 0 else ("base", "new")
        dumps = {}
        for b in order:
            dumps[b] = os.path.join(tmp, "%s_%d.npz" % (b, r))
            env = dict(os.environ, CM_LIB_PATH=libs[b])
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--seconds", str(a.seconds), "--filters", a.filters,
                                "--child", inputs, dumps[b]], env=env, capture_output=True, text=True)
            if p.returncode != 0:
                sys.stderr.write(p.stdout + p.stderr)
                raise SystemExit("the %s build failed in round %d" % (b, r))
            for k, ts in json.loads(p.stdout.strip().splitlines()[-1]).items():
                per.setdefault(k, {}).setdefault(b, []).append(float(np.median(ts)))
        x, y = np.load(dumps["new"]), np.load(dumps["base"])
        if sorted(x.files) != sorted(y.files):
            res["mismatches"].append("round %d: different output sets" % r)
        for k in x.files:
            if k in y.files and not np.array_equal(x[k], y[k]):
                res["mismatches"].append("round %d: %s" % (r, k))
        res["rounds_done"] = r + 1
        worst = summarize(res, per, out)
    for k, row in res["cases"].items():
        print("%-70s new %9.3f +- %7.3f  base %9.3f +- %7.3f  %s" % (
            k, row["new"]["median_ms"], row["new"]["spread_ms"], row["base"]["median_ms"], row["base"]["spread_ms"],
            "SLOWER" if row["slower_than_spread"] else ""))
    print(json.dumps({"gpu": res["gpu"], "bit_identical": res["bit_identical"], "mismatches": res["mismatches"][:10],
                      "n_cases": len(res["cases"]), "n_slower_than_spread": res["n_slower_than_spread"],
                      "worst_relative_change": round(worst, 4), "out": out}))


if __name__ == "__main__":
    main()
