#!/usr/bin/env python
"""BASELINE config 4: VoxelGrid of one aggregated map cloud partitioned over the GPUs of one box by voxel-key range, with
one NCCL all-to-all -- cm_giant_voxelgrid, C++ + NCCL behind the C ABI. Launch with torchrun (one rank per GPU) or plainly
for one GPU.
Prints one JSON line on rank 0. --check compares against the CPU oracle (small clouds only)."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cloud_merger_b200 import CloudMerger, GiantCloud, giant_unique_id, synth  # noqa: E402


def main():
    # one JSON line on stdout: whatever libraries print there (NCCL's version banner) goes to stderr instead
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=100_000_000)
    ap.add_argument("--leaf", type=float, default=0.02)
    ap.add_argument("--min-points", type=int, default=1)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--nan-every", type=int, default=0, help="K > 0: every K-th point gets a NaN y (non-finite rows, which stay on their rank)")
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--stages", action="store_true", help="one more (profiled, blocking) call after the timed ones: device time per stage")
    a = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n = a.points
    lo, hi = rank * n // world, (rank + 1) * n // world
    # every rank generates the same cloud chunk-wise and keeps its block (deterministic, no host exchange)
    whole = synth.map_cloud(4, n)
    if a.nan_every > 0:
        whole[::a.nan_every, 1] = np.nan
    local = torch.from_numpy(np.ascontiguousarray(whole[lo:hi])).cuda()
    if not a.check:
        whole = None
    # capacity: a rank may receive more than its share
    cap = int(min(n, (hi - lo) * 2 + 1024))
    cm = CloudMerger(device=local_rank, max_batch_points=cap)
    cm.set_voxel(a.leaf, a.min_points, True)
    # the product path: the whole partitioned VoxelGrid behind the C ABI (C++ + NCCL inside the library). torch only ships
    # the 128-byte NCCL id to the ranks and holds the input tensor.
    nccl_id = None
    if world > 1:
        box = [giant_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        nccl_id = box[0]
    giant = GiantCloud(cm, rank, world, nccl_id)
    stream = torch.cuda.current_stream().cuda_stream
    times, out = [], None
    for it in range(a.iters + 1):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = giant.voxelgrid(local.data_ptr(), int(local.shape[0]), stream=stream)
        st = cm.stats()   # blocks until the voxels are there
        if world > 1:
            dist.barrier()
        if it:
            times.append(time.perf_counter() - t0)
    stage_ms = None
    if a.stages:
        cm.set_profiling(True)
        if world > 1:
            dist.barrier()
        stage_ms = giant.voxelgrid(local.data_ptr(), int(local.shape[0]), stream=stream)["stage_ms"]
        st = cm.stats()
        cm.set_profiling(False)
    out.update(n_voxels=int(st.voxels_out), gpu_ms=float(st.gpu_ms), key_bits=int(st.key_bits))
    if a.check:
        o = cm.device_out()
        v = out["n_voxels"]
        out.update(idx=cm.download(o.voxel_idx, np.uint64, v).astype(np.int64), count=cm.download(o.voxel_count, np.uint32, v),
                   centroid=cm.download(o.voxel_xyzi, np.float32, v * 4).reshape(v, 4))
    dt = float(np.median(times))
    stats = torch.tensor([out["points_received"], out["points_sent_away"], out["n_voxels"]], dtype=torch.int64, device="cuda")
    if world > 1:
        allv = [torch.zeros_like(stats) for _ in range(world)]
        dist.all_gather(allv, stats)
    else:
        allv = [stats]
    check = None
    if a.check:
        from oracle import cm_oracle_py as oracle
        gathered = [None] * world
        mine = (rank, out["idx"], out["count"], out["centroid"])
        if world > 1:
            dist.all_gather_object(gathered, mine)
        else:
            gathered = [mine]
        if rank == 0:
            gathered.sort(key=lambda t: t[0])
            idx = np.concatenate([g[1] for g in gathered]); cnt = np.concatenate([g[2] for g in gathered])
            cen = np.concatenate([g[3] for g in gathered])
            o = oracle.voxelgrid(whole, [a.leaf] * 3, a.min_points, True, force64=True, is_dense=a.nan_every <= 0)
            ok = len(idx) == o["n"] and (idx == o["idx"]).all() and (cnt == o["count"]).all()
            ok = ok and (cen.view(np.uint32) == o["centroid"].view(np.uint32)).all()   # bit-equal to the float oracle
            rel = np.abs(cen - o["centroid_f64"]) / np.maximum(np.abs(o["centroid_f64"]), 1e-2)
            ok = ok and rel.max() <= 1e-5
            check = "ok" if ok else "MISMATCH"
    if rank == 0:
        sent = int(sum(int(v[1]) for v in allv))
        os.write(real_stdout, (json.dumps({"workload": "cfg4: %d-pt map cloud, VoxelGrid %.3f m, key-range partition + all-to-all" % (n, a.leaf),
                          "n_gpus": world, "points": n, "voxels": int(sum(int(v[2]) for v in allv)), "ms": dt * 1e3,
                          "mpoints_per_s": n / dt / 1e6, "points_exchanged": sent, "bytes_exchanged": sent * 16,
                          "points_per_rank_after": [int(v[0]) for v in allv], "key_bits": out.get("key_bits"),
                          "local_voxelgrid_ms": out.get("gpu_ms"), "host_syncs_before_report": out.get("host_syncs"),
                          "exchange": out.get("exchange"),
                          "stage_ms_rank0": dict(zip(["plan", "group", "exchange", "voxelgrid"], stage_ms)) if stage_ms else None,
                          "api": "cm_giant_voxelgrid (C++ + NCCL behind the C ABI)", "check": check}) + "\n").encode())
    giant.close()
    cm.close()
    if world > 1:
        dist.destroy_process_group()
    return 0 if check in (None, "ok") else 1


if __name__ == "__main__":
    sys.exit(main())
