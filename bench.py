#!/usr/bin/env python
"""bench.py -- merged + voxel-filtered Mpoints/s of the merge hot path (BASELINE.json metric) on N B200s.

A step = one pass of the whole hot path (transform -> concat -> crop -> VoxelGrid) over one batch of F frames of the
named workload (default: BASELINE config 3, 8 sensors x 256k points per frame, box crop, VoxelGrid 0.05 m -- the config
BASELINE.json names for 1/2/4/8 GPUs; frames are sharded over the ranks with no collective).
  value    device-resident throughput: inputs already in HBM, CUDA-event timed, max over ranks
  e2e      the same metric through the host C-ABI path (cm_submit_cloud_pinned / cm_merge_frame_async / cm_wait_frame)
           from pinned HOST buffers, H2D and D2H inside the timed region
  roofline the dominant kernel's algorithmic bytes / its CUDA-event duration against MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle (port of the PCL 1.8.1 path; the reference's own PCL build is not installable here)
--impl reference times that CPU path alone, on all host cores, for the driver's own ratio.
--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy, so that two builds can be compared.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True   # the tree may be read-only: nothing is written next to the sources
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "merged+voxel-filtered Mpoints/s"
UNIT = "Mpoints/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"],
                    help="BASELINE.json config; cfg3 (8 x 256k points per frame, frame-sharded) is the 1/2/4/8-GPU config")
    ap.add_argument("--frames", type=int, default=0, help="frames per step (0 = enough to exceed L2 several times)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-path measurement (0 = min(steps, 3))")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-latency", action="store_true", help="skip the single-frame p50/p99 latency measurement")
    ap.add_argument("--points", type=int, default=0, help="cfg4 / cfg5: points of the cloud (0 = 100 M / 16 Mi)")
    ap.add_argument("--sustained-seconds", type=float, default=0.0,
                    help="length of an extra back-to-back leg that shows the number holds at steady-state clocks (0 = skip, "
                         "the default: then --steps is the number of timed steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed (on rank 0) to DIR/<name>.npy (frame workloads cfg1-cfg3)")
    return ap.parse_args()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe). The timed region of this
    workload lasts milliseconds, so the primary source is an NVML polling thread (one sample per ~2 ms); nvidia-smi -lms
    (one sample per 100 ms at best) runs beside it as the recipe's own view and is merged in."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, uuid: str = ""):
        self.gpu = gpu_index
        self.uuid = uuid
        self.rows = []
        self.proc = None
        self.nv = []        # (sm_mhz, reasons bitmask)
        self.nv_max = None
        self._stop = threading.Event()
        self._thr = None
        self._nvml = None
        self._nvml_open()

    def _nvml_open(self):
        """NVML handle of this rank's GPU, opened before the timed region (nvmlInit takes milliseconds)."""
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = None
            if self.uuid:
                for cand in (self.uuid, "GPU-" + self.uuid):
                    try:
                        h = nv.nvmlDeviceGetHandleByUUID(cand.encode() if isinstance(cand, str) else cand)
                        break
                    except Exception:
                        h = None
            if h is None:
                h = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            self.nv_max = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self._nvml = (nv, h)
        except Exception as e:  # keep going on nvidia-smi alone, but say why
            self._nvml = None
            print("[bench] NVML sampling unavailable: %r" % (e,), file=sys.stderr)

    def _nvml_loop(self):
        if not self._nvml:
            return
        nv, h = self._nvml

        def get_reasons(hh):
            for name in ("nvmlDeviceGetCurrentClocksEventReasons", "nvmlDeviceGetCurrentClocksThrottleReasons"):
                fn = getattr(nv, name, None)
                if fn is not None:
                    try:
                        return int(fn(hh))
                    except Exception:
                        continue
            return 0
        try:
            while not self._stop.is_set():
                self.nv.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), get_reasons(h)))
                time.sleep(0.001)
        except Exception as e:
            print("[bench] NVML sampling stopped: %r" % (e,), file=sys.stderr)

    def start(self):
        self._thr = threading.Thread(target=self._nvml_loop, daemon=True)
        self._thr.start()
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=1.0)
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        # NVML bit masks: 0x8 hw_slowdown, 0x40 hw_thermal_slowdown, 0x20 sw_thermal_slowdown, 0x4 sw_power_cap
        for clk, bits in self.nv:
            sm.append(clk)
            for name, bit in (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)):
                if bits & bit:
                    reasons.add(name)
        if self.nv_max:
            mx.append(self.nv_max)
        n_nvml = len(sm)
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvml x%d + nvidia-smi x%d" % (n_nvml, len(sm) - n_nvml)}


def dram_traffic(kernel: str, workload: str, frames: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed `ncu --set full` capture of
    this same workload (profiles/traffic.json, written by scripts/ncu_traffic.py); None when no capture matches."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        e = d.get("%s/%d" % (workload, frames), {}).get(kernel)
        return int(e["bytes_per_launch"]) if e else None
    except Exception:
        return None


def workload_spec(name: str, frames: int):
    from cloud_merger_b200 import synth
    c = dict(synth.CONFIGS[name])
    n = c["rings"] * c["azimuth"]
    if frames <= 0:
        # >= 4x the 126 MB L2 of raw input per step, so every step streams from HBM
        frames = max(1, int(np.ceil(4 * 126e6 / (c["sensors"] * n * 16))))
        frames = min(frames, 64)
    c.update(points_per_sensor=n, frames=frames)
    return c


def make_host_frames(spec, name: str, rank: int, pinned: bool):
    """F distinct synthetic frames (new noise per frame), packed 16-byte xyzi records, one buffer per (frame, sensor)."""
    from cloud_merger_b200 import host_alloc, synth
    S, n, F = spec["sensors"], spec["points_per_sensor"], spec["frames"]
    seed = 1000 * int(name[-1])
    nbytes = n * 16
    if pinned:
        arena, addr = host_alloc(F * S * nbytes)
    else:
        arena, addr = np.empty(F * S * nbytes, np.uint8), 0
    bufs = []
    for f in range(F):
        row = []
        for s in range(S):
            off = (f * S + s) * nbytes
            view = arena[off:off + nbytes].view(np.float32).reshape(n, 4)
            view[:] = synth.lidar_cloud(seed, s, rank * 100000 + f, spec["rings"], spec["azimuth"])
            row.append((view, (addr + off) if pinned else view.ctypes.data))
        bufs.append(row)
    return arena, bufs


DUMP_ROWS = 1 << 18


def dump_outputs(cm, out_dir: str):
    """--dump-outputs: the results the last cm_run_batch left for its caller, as .npy files in float32 / float64.
    frame_info: one row per frame (survivor_begin, survivor_end, voxel_begin, voxel_end, min_b[3], max_b[3], div_b[3],
    pcl_overflow). survivor_xyzi / survivor_src and voxel_xyzi / voxel_count / voxel_idx: the same DUMP_ROWS rows of each
    kind, drawn with a fixed seed from its count (all rows when there are fewer), which keeps the dump near 15 MB."""
    r = cm.fetch_batch_outputs(want_sorted=False)
    arrays = {"frame_info": np.array([[f.survivor_begin, f.survivor_end, f.voxel_begin, f.voxel_end, *f.min_b, *f.max_b,
                                       *f.div_b, f.pcl_overflow] for f in r["frames"]], np.float64)}
    for kind, fields in (("survivor", ("xyzi", "src")), ("voxel", ("xyzi", "count", "idx"))):
        n = len(r[kind + "_xyzi"])
        rows = np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_ROWS), replace=False))
        for f in fields:
            a = r[kind + "_" + f][rows]
            arrays[kind + "_" + f] = a if a.dtype == np.float32 else a.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_port(spec, host_frames, seconds: float, threads_frames: int, sensor_threads: int):
    """Times the CPU oracle (port of the reference's PCL path) on a bounded sample of the same frames."""
    from concurrent.futures import ThreadPoolExecutor

    from cloud_merger_b200 import synth
    from oracle import cm_oracle_py as oracle
    S = spec["sensors"]
    mats = [synth.extrinsic(s, S)[:3].reshape(-1) for s in range(S)]

    def one(f):
        cds = [dict(data=host_frames[f][s][0].view(np.uint8).reshape(-1), n_points=spec["points_per_sensor"], point_step=16,
                    off_x=0, off_y=4, off_z=8, off_i=12, is_dense=1, m=mats[s]) for s in range(S)]
        r = oracle.merge_frame(cds, spec["passes"], [spec["leaf"]] * 3, spec["min_points"], True, True,
                               threads=sensor_threads, want_outputs=False)
        return r["n_voxels"]

    F = len(host_frames)
    one(0)  # warm-up (page faults, library load)
    done, t0 = 0, time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads_frames) as ex:
        while True:
            batch = [(done + i) % F for i in range(threads_frames)]
            list(ex.map(one, batch))
            done += len(batch)
            if time.perf_counter() - t0 >= seconds:
                break
    dt = time.perf_counter() - t0
    pts = done * S * spec["points_per_sensor"]
    return pts / dt / 1e6, done, dt


def run_reference(args):
    """The reference arm: the reference's own CPU implementation of the path. PCL/ROS cannot be installed here
    (SURVEY.md section 8c), so this is the oracle port, run frame-parallel on every host core."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    spec = workload_spec(args.workload, args.frames)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    # one frame per thread and at least one thread per core the process may use: every host core is busy in every step
    sample_frames = max(4, min(64, max(spec["frames"], cores)))
    spec_small = dict(spec, frames=sample_frames)
    _, frames = make_host_frames(spec_small, args.workload, 0, pinned=False)
    from concurrent.futures import ThreadPoolExecutor

    from cloud_merger_b200 import synth
    from oracle import cm_oracle_py as oracle
    S = spec["sensors"]
    mats = [synth.extrinsic(s, S)[:3].reshape(-1) for s in range(S)]

    def one(f):
        cds = [dict(data=frames[f][s][0].view(np.uint8).reshape(-1), n_points=spec["points_per_sensor"], point_step=16,
                    off_x=0, off_y=4, off_z=8, off_i=12, is_dense=1, m=mats[s]) for s in range(S)]
        return oracle.merge_frame(cds, spec["passes"], [spec["leaf"]] * 3, spec["min_points"], True, True, threads=1,
                                  want_outputs=False)["n_voxels"]

    workers = min(cores, sample_frames)
    with ThreadPoolExecutor(max_workers=workers) as ex:
        def step():
            list(ex.map(one, range(sample_frames)))
        for _ in range(args.warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        dt = time.perf_counter() - t0
    pts_step = sample_frames * S * spec["points_per_sensor"]
    value = pts_step * args.steps / dt / 1e6
    sample = "%d frames/step of %s, frame-parallel on %d threads (oracle port of the PCL 1.8.1 path)" % (
        sample_frames, args.workload, workers)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%s: %s" % (args.workload, spec["what"]), "frames_per_step": sample_frames,
                   "points_per_frame": S * spec["points_per_sensor"], "leaf_m": spec["leaf"],
                   "min_points": spec["min_points"], "crop": spec["passes"]},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


CLOUD_WORKLOADS = {
    "cfg4": dict(points=100_000_000, leaves=[0.02], min_points=1,
                 what="single 100M-pt aggregated map cloud VoxelGrid 0.02 m, voxel-key range partition + one NCCL all-to-all"),
    "cfg5": dict(points=1 << 24, leaves=[0.01, 0.02, 0.05, 0.1, 0.2, 0.5, 1.0], min_points=1,
                 what="VoxelGrid leaf-size sweep 0.01-1.0 m on 16 Mi pts (uniform 200 x 200 x 10 m)"),
}


def cloud_of(name: str, n: int, rank: int, world: int):
    """This rank's block of the workload's cloud (cfg4: every rank generates the seeded map and keeps its block)."""
    from cloud_merger_b200 import synth
    if name == "cfg5":
        return synth.uniform_cloud(5000, n)
    whole = synth.map_cloud(4, n)
    lo, hi = rank * n // world, (rank + 1) * n // world
    return np.ascontiguousarray(whole[lo:hi])


def run_cloud_reference(args):
    """--impl reference for cfg4 / cfg5: the oracle's VoxelGrid (port of PCL 1.8.1's, 64-bit index extension) on a bounded
    sample of the cloud, one leaf per thread."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    from concurrent.futures import ThreadPoolExecutor

    from oracle import cm_oracle_py as oracle
    wl = CLOUD_WORKLOADS[args.workload]
    n = min(args.points or wl["points"], 4_000_000)
    x = cloud_of(args.workload, n, 0, 1)
    cores = os.cpu_count() or 1
    jobs = wl["leaves"] if len(wl["leaves"]) > 1 else wl["leaves"] * min(cores, 4)
    workers = min(cores, len(jobs))

    def one(leaf):
        return oracle.voxelgrid(x, [leaf] * 3, wl["min_points"], True, force64=True)["n"]
    with ThreadPoolExecutor(max_workers=workers) as ex:
        for _ in range(min(args.warmup, 1)):
            list(ex.map(one, jobs))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            list(ex.map(one, jobs))
        dt = time.perf_counter() - t0
    value = n * len(jobs) * args.steps / dt / 1e6
    sample = "%d-point sample, %d VoxelGrid runs per step on %d threads (oracle port of PCL 1.8.1 VoxelGrid, 64-bit index)" % (n, len(jobs), workers)
    emit({"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
          "scaling": "strong" if args.workload == "cfg4" else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
          "config": {"workload": "%s: %s" % (args.workload, wl["what"]), "points": n, "leaves_m": wl["leaves"]},
          "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port", "sample": sample},
          "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0})
    return 0


def run_cloud_workload(args):
    """cfg4 (one giant cloud, partitioned over the ranks: cm_giant_voxelgrid, strong scaling) and cfg5 (leaf sweep on one
    cloud per GPU; N > 1 = independent replicas). A step = the VoxelGrid of the cloud at every leaf of the workload."""
    import torch
    import torch.distributed as dist

    from cloud_merger_b200 import CloudMerger, GiantCloud, giant_unique_id, host_alloc
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    wl = CLOUD_WORKLOADS[args.workload]
    giant_mode = args.workload == "cfg4"
    n_total = args.points or wl["points"]
    local = cloud_of(args.workload, n_total, rank if giant_mode else 0, world if giant_mode else 1)
    n = len(local)
    pinned, addr = host_alloc(n * 16)
    pinned[:] = local.view(np.uint8).reshape(-1)
    cap = n if not giant_mode or world == 1 else int(min(n_total, 2 * n + 1024))
    cm = CloudMerger(device=local_rank, max_batch_points=cap)
    dev = cm.device_buffer(n * 16)
    dev.upload(local)
    stream = torch.cuda.current_stream().cuda_stream
    giant = None
    if giant_mode:
        nccl_id = None
        if world > 1:
            box = [giant_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            nccl_id = box[0]
        giant = GiantCloud(cm, rank, world, nccl_id)
    cm.set_profiling(True)
    leaves = wl["leaves"]
    per_leaf = {}

    def one_leaf(leaf, record=False):
        cm.set_voxel(leaf, wl["min_points"], True)
        if giant:
            info = giant.voxelgrid(dev.ptr, n, stream=stream)
        else:
            info = {}
            cm.dev_voxelgrid(dev.ptr, n, stream=stream)
        if record:
            st = cm.stats()
            per_leaf[leaf] = dict(st=st, info=info, sort_ms=cm.stage_ms("sort"), key_ms=cm.stage_ms("key_hist"),
                                  cent_ms=cm.stage_ms("centroid"), launches=cm.launch_count())
        return info

    def step(record=False):
        for leaf in leaves:
            one_leaf(leaf, record)
    for _ in range(max(args.warmup, 3)):
        step()
        cm.sync()
    try:
        gpu_uuid = str(torch.cuda.get_device_properties(torch.cuda.current_device()).uuid)
    except Exception:
        gpu_uuid = ""
    sampler = ClockSampler(local_rank, gpu_uuid)
    barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for k in range(args.steps):
        step(record=(k == args.steps - 1))
    ev1.record()
    cm.sync()
    barrier()
    clocks = sampler.stop()
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    pts_job = (n_total if giant_mode else n * world) * len(leaves)
    value = pts_job * args.steps / (ms_total / 1e3) / 1e6
    peak, peak_src = peaks()
    stages, sort_bytes, sort_ms, sort_launches, launches = {}, 0, 0.0, 0, 0
    for leaf, r in per_leaf.items():
        st = r["st"]
        M, V, P, kb = int(st.points_in), int(st.voxels_out), int(st.sort_passes), int(st.key_bytes)
        b_vg = M * (16 + 2 * kb + 2 * P * (kb + 4) + (kb + 4) + 16) + 20 * V
        b_io = 16 * M + 20 * V
        ms = float(st.gpu_ms)
        stages["leaf_%g" % leaf] = {"ms": round(ms, 4), "points": M, "voxels": V, "key_bytes": kb, "passes": P, "key_bits": int(st.key_bits),
                                    "B_vg_bytes": int(b_vg), "frac": round(b_vg / (ms * 1e-3) / 1e9 / peak, 4) if ms > 0 else 0,
                                    "B_io_bytes": int(b_io), "frac_io": round(b_io / (ms * 1e-3) / 1e9 / peak, 4) if ms > 0 else 0,
                                    "pcl_could_run": not bool(st.pcl_overflow), "sort_ms": round(r["sort_ms"], 4),
                                    "key_hist_ms": round(r["key_ms"], 4), "centroid_ms": round(r["cent_ms"], 4)}
        if r["info"]:
            stages["leaf_%g" % leaf].update(points_received=r["info"]["points_received"], points_sent_away=r["info"]["points_sent_away"],
                                            bytes_sent=r["info"]["points_sent_away"] * 16)
        sort_bytes += M * 2 * (kb + 4) * P
        sort_ms += r["sort_ms"]
        sort_launches += P
        launches += r["launches"]
    achieved = sort_bytes / (sort_ms * 1e-3) / 1e9 if sort_ms > 0 else 0.0
    roofline = {"bound": "hbm", "kernel": "k_onesweep_pass", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": None, "peak_source": peak_src,
                "launch_ms": round(sort_ms / max(sort_launches, 1), 4),
                "algorithmic_bytes_per_launch": int(sort_bytes / max(sort_launches, 1)), "share_of_step": round(sort_ms / ms_step, 3)}
    # ---- end to end: the block from page-locked host memory in, centroids + counts + voxel ids out, every step ------------
    e2e = None
    if not args.no_e2e:
        e2e_steps = args.e2e_steps or min(args.steps, 2)
        cm.set_profiling(False)
        out_pin, _ = host_alloc(cap * 28)
        h2d = d2h = 0

        def host_step(count):
            nonlocal h2d, d2h
            cm._check(cm._lib.cm_memcpy_h2d(cm._h, dev.ptr, addr, n * 16, stream))
            for leaf in leaves:
                one_leaf(leaf)
                st = cm.stats()
                o = cm.device_out()
                v = int(st.voxels_out)
                base = out_pin.ctypes.data
                cm._check(cm._lib.cm_memcpy_d2h(cm._h, base, o.voxel_xyzi, v * 16, stream))
                cm._check(cm._lib.cm_memcpy_d2h(cm._h, base + v * 16, o.voxel_count, v * 4, stream))
                cm._check(cm._lib.cm_memcpy_d2h(cm._h, base + v * 20, o.voxel_idx, v * 8, stream))
                if count:
                    d2h += v * 28
            if count:
                h2d += n * 16
        host_step(False)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            host_step(True)
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        e2e = {"value": pts_job * e2e_steps / dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(h2d / e2e_steps),
               "d2h_bytes_per_step": int(d2h / e2e_steps), "steps": e2e_steps, "ms_per_step": dt / e2e_steps * 1e3,
               "api": ("cm_giant_voxelgrid" if giant else "cm_dev_voxelgrid") + " between cm_memcpy_h2d of the block and cm_memcpy_d2h of the voxels"}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import cm_oracle_py as oracle
        ns = min(n, 4_000_000)
        t0 = time.perf_counter()
        done = 0
        while time.perf_counter() - t0 < args.cpu_seconds:
            oracle.voxelgrid(local[:ns], [leaves[done % len(leaves)]] * 3, wl["min_points"], True, force64=True)
            done += 1
        secs = time.perf_counter() - t0
        cpu = {"value": ns * done / secs / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": "%d VoxelGrid runs over the first %d points in %.1f s on one thread (PCL's VoxelGrid is single-threaded; oracle port)" % (done, ns, secs)}
    if rank == 0:
        emit({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
              "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if giant_mode else "weak", "vs_baseline": None,
              "dtype": "f32", "data": "synthetic",
              "config": {"workload": "%s: %s" % (args.workload, wl["what"]), "points": n_total, "points_per_gpu": n, "leaves_m": leaves,
                         "min_points": wl["min_points"],
                         "sharding": ("voxel-key range partition, one NCCL all-to-all (cm_giant_voxelgrid)" if giant_mode and world > 1
                                      else "single GPU" if world == 1 else "independent replicas, one cloud per GPU"),
                         "l2": "inputs larger than L2 (%.0f MB per GPU)" % (n * 16 / 1e6)},
              "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches * args.steps), "roofline": roofline, "stages": stages,
              "cpu_baseline": cpu})
    if giant:
        giant.close()
    cm.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


_REAL_STDOUT = None


def guard_stdout():
    """The contract is ONE JSON line on stdout. Libraries print there too (NCCL's version banner at NCCL_DEBUG=WARN, for
    one), so file descriptor 1 is pointed at stderr for the whole run and the line is written to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    args = parse_args()
    guard_stdout()
    if args.dump_outputs and (args.impl != "b200" or args.workload in CLOUD_WORKLOADS):
        raise SystemExit("bench.py: --dump-outputs writes the outputs of the GPU path of the frame workloads cfg1-cfg3")
    if args.impl == "reference":
        return run_cloud_reference(args) if args.workload in CLOUD_WORKLOADS else run_reference(args)
    if args.workload in CLOUD_WORKLOADS:
        return run_cloud_workload(args)

    import torch
    import torch.distributed as dist

    from cloud_merger_b200 import CloudMerger, make_layout, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    spec = workload_spec(args.workload, args.frames)
    S, n, F = spec["sensors"], spec["points_per_sensor"], spec["frames"]
    pts_step = F * S * n
    pinned_arena, host_frames = make_host_frames(spec, args.workload, rank, pinned=True)

    cm = CloudMerger(device=local_rank, max_sensors=S, max_points_per_sensor=n, max_point_step=16, frames_in_flight=4,
                     max_batch_points=pts_step, max_batch_frames=F)
    for s in range(S):
        cm.set_extrinsic(s, synth.extrinsic(s, S))
    cm.set_crop(spec["passes"])
    cm.set_voxel(spec["leaf"], spec["min_points"], True)
    layout = make_layout()

    # ---- device-resident inputs -------------------------------------------------------------------------------------
    dev = torch.empty(pts_step * 16, dtype=torch.uint8, device="cuda")
    dev.copy_(torch.from_numpy(pinned_arena), non_blocking=False)
    items = []
    for f in range(F):
        for s in range(S):
            items.append((dev.data_ptr() + (f * S + s) * n * 16, n, layout, s, f))
    segs = cm.make_segments(items)
    stream = torch.cuda.current_stream().cuda_stream
    cm.set_profiling(True)

    stage_names = ["transform_crop", "grid", "key_hist", "sort", "centroid"]
    stage_acc = {k: 0.0 for k in stage_names}
    for _ in range(max(args.warmup, 3)):
        cm.run_batch(segs, stream=stream)
        cm.sync()
    st = cm.stats()
    if st.device_error:
        raise SystemExit("device error %d" % st.device_error)

    try:
        gpu_uuid = str(torch.cuda.get_device_properties(torch.cuda.current_device()).uuid)
    except Exception:
        gpu_uuid = ""
    sampler = ClockSampler(local_rank, gpu_uuid)
    barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    # The K steps are enqueued back to back, as a consumer of device-resident batches would, and the host reads the
    # report (survivor / voxel counts, stage events) once at the end: the stage times are those of the last timed step.
    ev0.record()
    for _ in range(args.steps):
        cm.run_batch(segs, stream=stream)
    ev1.record()
    cm.sync()
    launches = cm.launch_count() * args.steps
    for k in stage_names:
        stage_acc[k] = cm.stage_ms(k) * args.steps
    pass0_ms = cm.stage_ms("sort_pass0")
    barrier()
    clocks = sampler.stop()
    ms_total = ev0.elapsed_time(ev1)
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = pts_step * world * args.steps / (ms_total / 1e3) / 1e6
    st = cm.stats()
    M, V, P, kb = int(st.survivors), int(st.voxels_out), int(st.sort_passes), int(st.key_bytes)
    if args.dump_outputs and rank == 0:
        dump_outputs(cm, args.dump_outputs)   # before any later leg overwrites the last timed step's outputs

    # ---- sustained leg: the same step back to back for >= --sustained-seconds (the K-step region above lasts milliseconds,
    # too short for the GPU to reach its steady-state power / clocks) ---------------------------------------------------------
    sustained = None
    if args.sustained_seconds > 0:
        cm.set_profiling(False)
        n_sus = max(args.steps, int(np.ceil(args.sustained_seconds * 1e3 / ms_step)))
        sampler2 = ClockSampler(local_rank, gpu_uuid)
        barrier()
        sampler2.start()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(n_sus):
            cm.run_batch(segs, stream=stream)
        s1.record()
        cm.sync()
        barrier()
        clocks2 = sampler2.stop()
        ts = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        sus_ms = float(ts.item())
        sustained = {"steps": n_sus, "gpu_launches": int(cm.launch_count() * n_sus), "seconds": sus_ms / 1e3, "ms_per_step": sus_ms / n_sus,
                     "value": pts_step * world * n_sus / (sus_ms / 1e3) / 1e6, "unit": UNIT, "clocks": clocks2}
        cm.set_profiling(True)

    # ---- roofline: algorithmic bytes per launch / CUDA-event duration of that launch ----------------------------------
    peak, peak_src = peaks()
    stage_ms = {k: v / args.steps for k, v in stage_acc.items()}
    # K1 writes the voxel keys itself (4 B per survivor, at the survivor's slot) when the crop box bounds the grid: there is
    # then no key kernel, and radix pass 0 reads 4-byte keys instead of 8-byte records
    fused_keys = stage_ms["key_hist"] < 0.01
    algo = {
        "transform_crop": pts_step * 16 + M * (24 if fused_keys else 20),
        "key_hist": M * (16 + kb + 4),
        "sort": M * (2 * (kb + 4) * P) - (4 * M if fused_keys else 0),
        "centroid": M * (kb + 4 + 16) + V * 28,
    }
    stages = {}
    for k in ("transform_crop", "key_hist", "sort", "centroid"):
        if k == "key_hist" and fused_keys:
            continue
        ms = stage_ms[k]
        gbs = algo[k] / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        stages[k] = {"ms": round(ms, 4), "algorithmic_bytes": int(algo[k]), "achieved_gbs": round(gbs, 1),
                     "frac": round(gbs / peak, 4), "launches": P if k == "sort" else 1}
    vg_ms = stage_ms["grid"] + stage_ms["key_hist"] + stage_ms["sort"] + stage_ms["centroid"]
    b_vg = M * (16 + 2 * kb + 2 * P * (kb + 4) + (kb + 4) + 16) + 20 * V   # SURVEY 8d named-pipeline traffic
    b_io = 16 * M + 20 * V
    stages["voxelgrid_end_to_end"] = {
        "ms": round(vg_ms, 4), "B_vg_bytes": int(b_vg), "achieved_gbs": round(b_vg / (vg_ms * 1e-3) / 1e9, 1) if vg_ms > 0 else 0,
        "frac": round(b_vg / (vg_ms * 1e-3) / 1e9 / peak, 4) if vg_ms > 0 else 0,
        "B_io_bytes": int(b_io), "frac_io": round(b_io / (vg_ms * 1e-3) / 1e9 / peak, 4) if vg_ms > 0 else 0,
        "key_bytes": kb, "passes": P}
    dom = max(("transform_crop", "key_hist", "sort", "centroid"), key=lambda k: stage_ms[k])
    dom_launches = P if dom == "sort" else 1
    dom_ms_launch = stage_ms[dom] / dom_launches
    dom_bytes_launch = algo[dom] / dom_launches
    achieved = dom_bytes_launch / (dom_ms_launch * 1e-3) / 1e9 if dom_ms_launch > 0 else 0.0
    roof_kernel = {"transform_crop": "k_transform_crop", "key_hist": "k_voxel_key_hist", "sort": "k_onesweep_pass",
                   "centroid": "k_voxel_centroid"}[dom]
    roofline = {"bound": "hbm", "kernel": roof_kernel,
                "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": dram_traffic(roof_kernel, args.workload, F), "peak_source": peak_src, "launch_ms": round(dom_ms_launch, 4),
                "algorithmic_bytes_per_launch": int(dom_bytes_launch), "share_of_step": round(stage_ms[dom] / ms_step, 3)}
    if dom == "sort" and pass0_ms > 0 and P > 1:
        # the average above mixes two kinds of launch: pass 0 of a fused-key run reads the 4-byte keys through K1's tile records
        # and also counts the digits of the later passes (the work of the key kernel it replaced); passes 1.. are the plain pass
        b0 = M * (12 if fused_keys else 2 * (kb + 4))
        rest_ms = (stage_ms["sort"] - pass0_ms) / (P - 1)
        rest_b = M * 2 * (kb + 4)
        roofline["per_launch"] = {
            "pass0" + ("_fused_keys" if fused_keys else ""): {"ms": round(pass0_ms, 4), "algorithmic_bytes": int(b0),
                                                               "frac": round(b0 / (pass0_ms * 1e-3) / 1e9 / peak, 4)},
            "passes_1_to_%d" % (P - 1): {"ms": round(rest_ms, 4), "algorithmic_bytes": int(rest_b),
                                         "frac": round(rest_b / (rest_ms * 1e-3) / 1e9 / peak, 4) if rest_ms > 0 else None}}

    # ---- end to end through the host C-ABI path, pinned host buffers, H2D + D2H inside the timed region -----------------
    e2e = None
    if not args.no_e2e:
        e2e_steps = args.e2e_steps or min(args.steps, 3)
        cm.set_profiling(False)  # the stage events of the resident run are not wanted between the kernels of this path
        cap = S * n
        h2d = d2h = 0

        from cloud_merger_b200 import _lib as cm_lib
        view = cm_lib.CmFrameView()   # results are read in place: cm_wait_frame_view hands out the frame's page-locked mirrors

        # one call per frame hands over all S page-locked sensor clouds (adjacent in host memory: one 8 MB PCIe copy)
        submit = [cm.prepared_frame_submit(list(range(S)), [host_frames[f][s][1] for s in range(S)], [n] * S,
                                           [layout] * S, stamp=f) for f in range(F)]

        def host_step(count_bytes: bool):
            nonlocal h2d, d2h
            pending = []
            for f in range(F):
                submit[f]()
                pending.append(cm.merge_frame_async())
                if len(pending) >= 3:
                    cm.wait_frame_view(pending.pop(0), view)
                    if count_bytes:
                        d2h += view.n_voxels * 28
            while pending:
                cm.wait_frame_view(pending.pop(0), view)
                if count_bytes:
                    d2h += view.n_voxels * 28
            if count_bytes:
                h2d += F * S * n * 16

        host_step(False)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            host_step(True)
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        e2e = {"value": pts_step * world * e2e_steps / dt / 1e6, "unit": UNIT,
               "h2d_bytes_per_step": int(h2d / e2e_steps), "d2h_bytes_per_step": int(d2h / e2e_steps),
               "steps": e2e_steps, "ms_per_step": dt / e2e_steps * 1e3,
               "api": "cm_submit_clouds_pinned + cm_merge_frame_async + cm_wait_frame_view, 3 frames in flight; the voxels "
                      "(xyzi + count + idx, 28 B each) land in page-locked host memory on the frame's own stream"}

    # ---- single-frame latency (resident inputs) -----------------------------------------------------------------------
    latency = None
    if not args.no_latency and rank == 0:
        one = cm.make_segments(items[:S])
        lat = []
        for i in range(220):
            cm.run_batch(one, stream=stream)
            cm.sync()
            if i >= 20:
                lat.append(cm.stats().gpu_ms)
        lat.sort()
        latency = {"p50_ms": lat[len(lat) // 2], "p99_ms": lat[int(len(lat) * 0.99)], "frames": len(lat),
                   "what": "device time of one resident frame, first to last kernel"}
        if not args.no_e2e:
            # the same through the host path, nothing else in flight: page-locked clouds in -> voxels in host memory
            hl = []
            for i in range(120):
                f = i % F
                t0 = time.perf_counter()
                submit[f]()
                cm.wait_frame_view(cm.merge_frame_async(), view)
                if i >= 20:
                    hl.append((time.perf_counter() - t0) * 1e3)
            hl.sort()
            latency.update({"host_p50_ms": hl[len(hl) // 2], "host_p99_ms": hl[int(len(hl) * 0.99)],
                            "host_what": "wall time of one frame through cm_submit_clouds_pinned + merge + wait (%.0f MB in, voxels out)" % (S * n * 16 / 1e6)})

    # ---- CPU baseline on this box's host cores (rank 0, N = 1 only) ------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        sensor_threads = min(S, 6)
        v, frames_done, secs = cpu_port(spec, host_frames, args.cpu_seconds, 1, sensor_threads)
        cpu = {"value": v, "unit": UNIT, "cores": sensor_threads, "kind": "port",
               "sample": "%d frames of %s in %.1f s; per-sensor transform+crop on %d threads, concat+VoxelGrid on 1 "
                         "(mirrors AsyncSpinner(6) + main loop); oracle port, PCL itself is not installable here" % (
                             frames_done, args.workload, secs, sensor_threads)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "%s: %s" % (args.workload, spec["what"]), "frames_per_step": F,
                       "points_per_frame": S * n, "points_per_step_per_gpu": pts_step, "leaf_m": spec["leaf"],
                       "min_points": spec["min_points"], "crop": spec["passes"], "survivors_per_step": M,
                       "voxels_per_step": V, "key_bytes": kb, "sort_passes": P, "key_bits": int(st.key_bits),
                       "keys_from": "k_transform_crop (crop-box grid)" if fused_keys else "k_voxel_key_hist",
                       "sharding": "frames round-robin over ranks, no collective",
                       "timed_region": "K steps enqueued back to back on one stream, one report read at the end; stage times = last timed step",
                       "l2": "inputs larger than L2 (%.0f MB raw input per step per GPU)" % (pts_step * 16 / 1e6)},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "stages": stages,
            "cpu_baseline": cpu, "sustained": sustained,
        }
        if latency:
            line["latency"] = latency
        emit(line)
    cm.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
