"""Device-resident mirror of one main-loop iteration of the reference's built node `pcl_preprocessing`
(pcl_preprocessing/src/pc_preprocessing_main.cpp):

    callbackX      :318-470   pcl_ros::transformPointCloud into base_footprint, then proceedX
    proceedX       :228-312   getROI, five x windows (getCloudPart), per window removeGround:
    removeGround   :71-122      two z windows, RANSAC plane + ExtractIndices, outlierRemoval of what is not ground,
                                the points above the window appended
    fusePointclouds:131-160   no_ground / ground clouds of all sensors appended in sensor order
    voxelgrid      :168-177   VoxelGrid of the fused no_ground cloud

Everything between the upload of the raw sensor clouds and the download of the three published clouds stays in device
memory. The stages are the C-ABI calls of include/cloud_merger_gpu.h: transform + ROI crop of all sensors in one launch
(frame = sensor), per sensor ONE call for the whole proceedX body (cm_dev_proceed_zones: one zone-slicing pass, one
multi-cloud plane search, one multi-cloud radius outlier removal, the appends), device-to-device appends of the sensors,
one VoxelGrid. The per-sensor calls run concurrently -- one host thread, one handle and one CUDA stream per sensor, as the
reference's callbacks do on ros::AsyncSpinner(6) (pc_preprocessing_main.cpp:513). The C++ counterpart is
cloud_merger::PreprocessingFrame in include/cloud_merger_shim.hpp.

Host glue, not a kernel: there is no CPU fallback and no arithmetic on points here.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .api import ROI_PASSES, CloudMerger, make_layout

# {length, deviation, z_max_ground} per x window, front to rear: Parameter.h:45-55 with roi_mid = 15 (proceedFront)
FRONT_PARTS = ((30.0, 30.0, 2.5), (11.0, 19.0, 2.0), (15.0, 4.0, 1.5), (8.0, -4.0, 0.3), (11.0, -15.0, 0.5))


def zones_of_parts(parts, roi_z_max: float):
    """The PassThrough chains getCloudPart + removeGround run per x window: first all ground windows
    (x in [dev, dev + len], z in [-zg, zg]), then all upper windows (z in [zg + 0.01, roi_z_max]; `+ 0.01` is the reference's
    double sum narrowed to float by setFilterLimits)."""
    low, high = [], []
    for (length, dev, zg) in parts:
        x = (0, float(np.float32(dev)), float(np.float32(np.float32(dev) + np.float32(length))), 0)
        zf = np.float32(zg)
        low.append([x, (2, float(-zf), float(zf), 0)])
        high.append([x, (2, float(np.float32(np.float64(zf) + 0.01)), float(np.float32(roi_z_max)), 0)])
    return low + high


@dataclass
class NodeParams:
    """Parameter.h of pcl_preprocessing (:23-42)."""
    roi_passes: Sequence[Tuple[int, float, float, int]] = tuple(ROI_PASSES)
    roi_z_max: float = 3.0
    voxel_size: float = 0.1
    points_per_voxel: int = 2
    radius: float = float(np.float32(0.15))
    min_neighbor: int = 1
    max_iterations: int = 1000
    distance_threshold: float = float(np.float32(0.3))
    prob: float = float(np.float32(0.99))
    sum_order: int = 0
    # seg.setModelType / setAxis / setEpsAngle: the reference's SACMODEL_PLANE ignores the other two; with
    # CM_SAC_PERPENDICULAR_PLANE (1) only planes within eps_angle [rad] of horizontal count as ground
    sac_model: int = 0
    axis: Tuple[float, float, float] = (0.0, 0.0, 1.0)
    eps_angle: float = 0.0
    parts: Sequence[Sequence[Tuple[float, float, float]]] = field(default_factory=lambda: [FRONT_PARTS])  # per sensor (cycled)


class _SensorLane:
    """The proceedX body of one sensor: ONE handle, ONE C call (cm_dev_proceed_zones), its own CUDA stream -- one callback
    thread of the reference (ros::AsyncSpinner(6), pc_preprocessing_main.cpp:513)."""

    def __init__(self, device: int, max_points: int, p: NodeParams, parts):
        self.p = p
        self.parts = [tuple(pt) for pt in parts]
        self.h = CloudMerger(device=device, max_sensors=1, max_points_per_sensor=max_points, max_batch_points=max_points,
                             max_batch_frames=8)
        self.stream = self.h.stream_create()
        self.n_ng = self.n_g = 0
        self.no_ground_ptr = self.ground_ptr = 0
        self.planes: List[dict] = []

    def close(self):
        self.h.stream_destroy(self.stream)
        self.h.close()

    def run(self, roi_ptr: int, n: int):
        p = self.p
        r = self.h.dev_proceed_zones(roi_ptr, n, self.parts, p.roi_z_max, p.radius, p.min_neighbor, p.distance_threshold, p.prob,
                                     p.max_iterations, True, 12345, p.sum_order, stream=self.stream, model=p.sac_model,
                                     axis=p.axis, eps_angle=p.eps_angle)
        self.h.stream_sync(self.stream)
        self.n_ng, self.n_g = r["n_no_ground"], r["n_ground"]
        self.no_ground_ptr, self.ground_ptr = r["no_ground_ptr"], r["ground_ptr"]
        self.planes = r["planes"]


class PreprocessingNode:
    def __init__(self, n_sensors: int, max_points_per_sensor: int, params: Optional[NodeParams] = None, device: int = 0,
                 concurrent: bool = True):
        self.S = n_sensors
        self.p = params or NodeParams()
        self.concurrent = concurrent
        n = n_sensors * max_points_per_sensor
        mk = lambda frames: CloudMerger(device=device, max_sensors=n_sensors, max_points_per_sensor=max_points_per_sensor,
                                        max_batch_points=n, max_batch_frames=frames)
        self.crop = mk(n_sensors)   # transform + getROI of every sensor, one frame per sensor
        self.voxel = mk(1)
        self.crop.set_crop(self.p.roi_passes)
        self.voxel.set_voxel(self.p.voxel_size, self.p.points_per_voxel, True)
        self.raw = [self.crop.device_buffer(max_points_per_sensor * 16) for _ in range(n_sensors)]
        self.lanes = [_SensorLane(device, max_points_per_sensor, self.p, tuple(map(tuple, self.p.parts[s % len(self.p.parts)])))
                      for s in range(n_sensors)]
        self.no_ground = self.voxel.device_buffer(2 * n * 16)   # the fused clouds
        self.ground = self.voxel.device_buffer(2 * n * 16)
        self._pool = None
        if concurrent and n_sensors > 1:
            from concurrent.futures import ThreadPoolExecutor
            self._pool = ThreadPoolExecutor(max_workers=n_sensors)

    def close(self):
        if self._pool:
            self._pool.shutdown()
        for lane in self.lanes:
            lane.close()
        for h in (self.crop, self.voxel):
            h.close()

    def set_extrinsic(self, sensor: int, m: np.ndarray):
        self.crop.set_extrinsic(sensor, m)

    def frame(self, clouds: Sequence[np.ndarray], download: bool = True) -> dict:
        """clouds: one packed xyzi float32 array per sensor (sensor frame). Returns the three clouds the node publishes
        (/points_no_ground, /points_ground, /points_voxel) -- device pointers + sizes, and host copies when `download`."""
        items = []
        for s, c in enumerate(clouds):
            a = np.ascontiguousarray(c, np.float32).reshape(-1, 4)
            self.raw[s].upload(a)
            items.append((self.raw[s].ptr, len(a), make_layout(), s, s))
        self.crop.dev_transform_crop(self.crop.make_segments(items))
        self.crop.sync()
        info = self.crop.frame_info()
        roi = self.crop.device_out().survivor_xyzi
        # proceedX of every sensor: concurrently, one host thread + CUDA stream per sensor (the ctypes calls release the
        # GIL), or one after the other
        jobs = [(self.lanes[s], roi + info[s].survivor_begin * 16, info[s].survivor_end - info[s].survivor_begin)
                for s in range(len(clouds))]
        if self._pool:
            for f in [self._pool.submit(lane.run, ptr, n) for lane, ptr, n in jobs]:
                f.result()
        else:
            for lane, ptr, n in jobs:
                lane.run(ptr, n)
        # fusePointclouds: sensor after sensor
        n_ng = n_g = 0
        planes: List[dict] = []
        d2d = self.voxel.memcpy_d2d
        for lane, _, _ in jobs:
            d2d(self.no_ground.ptr + n_ng * 16, lane.no_ground_ptr, lane.n_ng * 16)
            d2d(self.ground.ptr + n_g * 16, lane.ground_ptr, lane.n_g * 16)
            n_ng += lane.n_ng
            n_g += lane.n_g
            planes += lane.planes
        self.voxel.dev_voxelgrid(self.no_ground.ptr, n_ng)
        self.voxel.sync()
        st = self.voxel.stats()
        vo = self.voxel.device_out()
        out = {"n_no_ground": n_ng, "n_ground": n_g, "n_voxels": int(st.voxels_out), "no_ground_ptr": self.no_ground.ptr,
               "ground_ptr": self.ground.ptr, "voxel_ptr": vo.voxel_xyzi, "planes": planes,
               "roi_points": [int(i.survivor_end - i.survivor_begin) for i in info[:len(clouds)]]}
        if download:
            out["no_ground"] = self.voxel.download(self.no_ground.ptr, np.float32, n_ng * 4).reshape(-1, 4)
            out["ground"] = self.voxel.download(self.ground.ptr, np.float32, n_g * 4).reshape(-1, 4)
            v = out["n_voxels"]
            out["voxel"] = self.voxel.download(vo.voxel_xyzi, np.float32, v * 4).reshape(-1, 4)
        return out
