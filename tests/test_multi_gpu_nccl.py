"""GPU tests of the giant-cloud mode (BASELINE config 4). The product path is cm_giant_voxelgrid -- C++ + NCCL behind the C
ABI: tested on one GPU at 20 M points against the oracle, on one GPU in "dry" mode (four virtual ranks: device-side grid,
histogram, splitters and grouping against the torch formulation of the gloo-tested host protocol), and on two ranks over
NCCL when the box has two GPUs. The building blocks (cm_set_voxel_bounds + cm_dev_voxelgrid, the routing kernels) keep their
own tests."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from cloud_merger_b200 import CloudMerger, multi_gpu, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_giant_backend_single_gpu(gpu_ok, oracle):
    import torch
    n, leaf, min_points = 400000, 0.1, 1
    whole = synth.map_cloud(7, n, extent=(120.0, 120.0, 10.0), n_boxes=100)
    whole[::1013, 1] = np.nan
    with CloudMerger(max_batch_points=n) as cm:
        pts = torch.from_numpy(whole).cuda()
        out = multi_gpu.giant_cloud_voxelgrid(pts, [leaf] * 3, min_points,
                                              multi_gpu.cuda_voxelgrid_backend(cm, leaf, min_points), 0, 1)
    o = oracle.voxelgrid(whole, [leaf] * 3, min_points, True, force64=True, is_dense=False)
    assert (out["idx"] == o["idx"]).all() and (out["count"] == o["count"]).all()
    assert (out["centroid"].view(np.uint32) == o["centroid"].view(np.uint32)).all()
    # bounds wider than the local cloud shift the grid origin exactly as a larger cloud would
    with CloudMerger(max_batch_points=n) as cm:
        cm.set_voxel(leaf, 1, True)
        lo = whole[np.isfinite(whole[:, :3]).all(axis=1), :3].min(axis=0) - np.float32(3.3)
        hi = whole[np.isfinite(whole[:, :3]).all(axis=1), :3].max(axis=0) + np.float32(1.7)
        cm.set_voxel_bounds(lo, hi)
        buf = cm.upload(whole)
        cm.dev_voxelgrid(buf.ptr, n, False)
        fi = cm.frame_info()[0]
    inv = np.float32(1.0) / np.float32(leaf)
    assert list(fi.min_b) == np.floor((lo * inv).astype(np.float32)).astype(int).tolist()


def test_cuda_router_pieces_single_gpu(gpu_ok):
    """The device-side routing steps against the torch formulation they replace: bounding box, key histogram and the
    grouping by key range (membership, source order inside a part, non-finite points to the local part)."""
    import torch
    n, leaf = 300000, 0.1
    whole = synth.map_cloud(9, n, extent=(100.0, 80.0, 8.0), n_boxes=80)
    whole[::997, 0] = np.nan
    whole[5::1999, 2] = np.inf
    pts = torch.from_numpy(whole).cuda()
    with CloudMerger(max_batch_points=n) as cm:
        cm.set_voxel(leaf, 1, True)
        router = multi_gpu.CudaRouter(cm, bins=4096)
        mn, mx, min_b, div_b = router.global_grid(pts, [leaf] * 3)
        t_mn, t_mx, t_min_b, t_div_b = multi_gpu.global_grid(pts, [leaf] * 3)
        assert (mn.view(np.uint32) == t_mn.view(np.uint32)).all() and (mx.view(np.uint32) == t_mx.view(np.uint32)).all()
        assert (min_b == t_min_b).all() and (div_b == t_div_b).all()
        keys = multi_gpu.voxel_keys(pts, [leaf] * 3, min_b, div_b)
        n_cells = int(div_b[0]) * int(div_b[1]) * int(div_b[2])
        hist = torch.zeros(4096, dtype=torch.int64, device="cuda")
        width = cm.dev_key_histogram(pts.data_ptr(), n, mn, mx, 4096, hist.data_ptr())
        assert width == max(1, -(-n_cells // 4096))
        want_hist = torch.bincount((keys[keys >= 0] // width).clamp_(0, 4095), minlength=4096)
        assert torch.equal(hist, want_hist)
        parts, me = 5, 2
        splitters = [n_cells * r // parts for r in range(1, parts)]
        cm.dev_route_by_key(pts.data_ptr(), n, mn, mx, splitters, me)
        got = cm.zone_out()
        dest = torch.searchsorted(torch.tensor(splitters, device="cuda"), keys, right=True)
        dest = torch.where(keys < 0, torch.full_like(dest, me), dest).cpu().numpy()
        assert len(got) == parts and sum(len(s) for _, s in got) == n
        for r in range(parts):
            want = np.nonzero(dest == r)[0]
            assert (got[r][1] == want).all(), "part %d" % r
            assert (got[r][0].view(np.uint32) == whole[want].view(np.uint32)).all()


def test_giant_c_abi_single_gpu_at_20m_points(gpu_ok, oracle):
    """cfg 4 at 20 M points on one GPU through cm_giant_voxelgrid (world 1: global grid on the device, key plan known from
    it, 64-bit keys on the big sort tile, 39 bits / 5 passes at leaf 0.02): voxel ids, counts, order bit-exact, centroids
    bit-equal to the float oracle and within 1e-5 of the float64 one."""
    from cloud_merger_b200 import GiantCloud
    n, leaf = 20_000_000, 0.02
    whole = synth.map_cloud(4000, n)
    with CloudMerger(max_batch_points=n) as cm:
        cm.set_voxel(leaf, 1, True)
        buf = cm.upload(whole)
        g = GiantCloud(cm, 0, 1)
        info = g.voxelgrid(buf.ptr, n)
        st = cm.stats()
        v = int(st.voxels_out)
        o_dev = cm.device_out()
        idx = cm.download(o_dev.voxel_idx, np.uint64, v).astype(np.int64)
        cnt = cm.download(o_dev.voxel_count, np.uint32, v)
        cen = cm.download(o_dev.voxel_xyzi, np.float32, v * 4).reshape(v, 4)
        g.close()
    o = oracle.voxelgrid(whole, [leaf] * 3, 1, True, force64=True)
    assert st.key_bytes == 8 and st.key_bits == info["key_bits"] > 32 and st.sort_passes == 5 and st.device_error == 0
    assert info["min_b"].tolist() == o["min_b"].tolist() and info["div_b"].tolist() == o["div_b"].tolist()
    assert v == o["n"] and (idx == o["idx"]).all() and (cnt == o["count"]).all()
    assert (cen.view(np.uint32) == o["centroid"].view(np.uint32)).all()
    err = np.abs(cen.astype(np.float64) - o["centroid_f64"]) / np.maximum(np.abs(o["centroid_f64"]), 1e-2)
    assert err.max() <= 1e-5


def test_giant_dry_routing_four_virtual_ranks(gpu_ok):
    """The device-side partition plan of cm_giant_voxelgrid without a communicator: grid, bin width, histogram, balancing
    splitters and the grouping by destination for four virtual ranks, against the torch formulation of the host protocol
    (multi_gpu.global_grid / voxel_keys / pick_splitters, which the gloo tests exercise on CPU)."""
    import torch
    from cloud_merger_b200 import GiantCloud
    n, leaf, world, me = 700000, 0.1, 4, 1
    whole = synth.map_cloud(11, n, extent=(150.0, 90.0, 9.0), n_boxes=120)
    whole[::991, 2] = np.nan
    pts = torch.from_numpy(whole).cuda()
    with CloudMerger(max_batch_points=n) as cm:
        cm.set_voxel(leaf, 1, True)
        g = GiantCloud(cm, me, world, None)
        info = g.voxelgrid(pts.data_ptr(), n, stream=torch.cuda.current_stream().cuda_stream)
        got = cm.zone_out()
        g.close()
    mn, mx, min_b, div_b = multi_gpu.global_grid(pts, [leaf] * 3)
    assert (info["min_p"].view(np.uint32) == mn.view(np.uint32)).all() and (info["max_p"].view(np.uint32) == mx.view(np.uint32)).all()
    assert (info["min_b"] == min_b).all() and (info["div_b"] == div_b).all()
    keys = multi_gpu.voxel_keys(pts, [leaf] * 3, min_b, div_b)
    n_cells = int(div_b[0]) * int(div_b[1]) * int(div_b[2])
    want_split = multi_gpu.pick_splitters(keys, n_cells, world, bins=1 << 14)
    assert info["splitters"] == want_split.cpu().tolist()
    assert info["points_total_finite"] == int((keys >= 0).sum().item())
    dest = torch.searchsorted(want_split.to(keys.device), keys, right=True)
    dest = torch.where(keys < 0, torch.full_like(dest, me), dest).cpu().numpy()
    assert len(got) == world and sum(len(s) for _, s in got) == n
    sizes = []
    for r in range(world):
        want = np.nonzero(dest == r)[0]
        assert (got[r][1] == want).all(), "part %d" % r
        assert (got[r][0].view(np.uint32) == whole[want].view(np.uint32)).all()
        sizes.append(len(want))
    assert info["send_begin"] == [0] + np.cumsum(sizes).tolist()
    assert info["points_sent_away"] == n - sizes[me]
    assert max(sizes) < 1.3 * n / world, "splitters balance the point counts (%r)" % sizes


@pytest.mark.parametrize("exchange", ["peer", "nccl", "peer-nonfinite"])
def test_giant_cloud_two_ranks_nccl(gpu_ok, exchange):
    """Two ranks, both exchanges: the grouping kernel storing into the peer's receive buffer over NVLink (the default
    where CUDA IPC maps the peers) and the grouped ncclSend / ncclRecv (CM_GIANT_NO_P2P=1); the merged voxels of both are
    checked against the oracle on the whole cloud. The non-finite case puts a NaN in every 997th point: at leaf 0.1 this
    cloud's index is 32 bits wide, so the sentinel frame of those points makes every rank's local key 33 bits."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, CM_GIANT_NO_P2P="1" if exchange == "nccl" else "0")
    port = {"peer": "29617", "nccl": "29619", "peer-nonfinite": "29621"}[exchange]
    extra = ["--nan-every", "997"] if exchange.endswith("nonfinite") else []
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", port,
                        os.path.join(ROOT, "scripts", "giant_cloud.py"),
                        "--points", "2000000", "--leaf", "0.1", "--check"] + extra, capture_output=True, text=True,
                       timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["check"] == "ok" and line["n_gpus"] == 2
    if exchange.endswith("nonfinite"):
        assert line["key_bits"] == 33
    if exchange == "nccl":
        assert line["exchange"] == "nccl"
    else:
        assert line["exchange"] in ("peer", "nccl")   # nccl where the box cannot map peers (no P2P between the devices)
