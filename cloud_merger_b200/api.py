"""Thin Python host layer over the C ABI (include/cloud_merger_gpu.h): used by the tests, bench.py and the multi-GPU
drivers. All compute happens in libcloud_merger_gpu.so on the GPU; nothing here computes on the CPU.

Names follow the reference's domain: clouds, sensors, extrinsics, crop passes (PassThrough), voxels, frames.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import (CM_MAX_ZONES, CM_MAX_ZONE_PASSES, CmConfig, CmCropBox, CmDeviceOut, CmFrameInfo, CmFrameOut, CmLayout,
                   CmPass, CmSegment, CmStats, CmZone, CmZoneOut)

# ---- layouts the reference's sensors produce (SURVEY.md section 8b) ------------------------------------------------------
LAYOUT_PACKED16 = dict(point_step=16, off_x=0, off_y=4, off_z=8, off_intensity=12)   # float4 x y z intensity
LAYOUT_PCL32 = dict(point_step=32, off_x=0, off_y=4, off_z=8, off_intensity=16)      # pcl::PointXYZI / Velodyne (Melodic)
LAYOUT_VELODYNE22 = dict(point_step=22, off_x=0, off_y=4, off_z=8, off_intensity=12)  # x y z intensity ring(u16) time(f32)
LAYOUT_LIVOX18 = dict(point_step=18, off_x=0, off_y=4, off_z=8, off_intensity=12)     # x y z reflectivity tag line

# getROI defaults, pcl_preprocessing/src/Parameter.h:31-35 (axis, lo, hi, negative)
ROI_PASSES = [(2, -0.5, 3.0, 0), (1, -5.0, 5.0, 0), (0, -15.0, 60.0, 0)]


IDENTITY_3X4 = (1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0)


def make_crop_box(min_pt, max_pt, translation=(0.0, 0.0, 0.0), rotation=(0.0, 0.0, 0.0), transform=IDENTITY_3X4,
                  negative: bool = False) -> CmCropBox:
    """One pcl::CropBox stage: setMin / setMax, setTranslation, setRotation (roll, pitch, yaw in rad), setTransform (3x4 or
    4x4 row-major; the identity is PCL's default) and setNegative."""
    t = np.asarray(transform, np.float32).reshape(-1)[:12]
    b = CmCropBox()
    for k in range(3):
        b.min[k] = float(np.float32(min_pt[k])); b.max[k] = float(np.float32(max_pt[k]))
        b.translation[k] = float(np.float32(translation[k])); b.rotation[k] = float(np.float32(rotation[k]))
    for k in range(12):
        b.transform[k] = float(t[k])
    b.negative = int(bool(negative))
    return b


class CloudMergerError(RuntimeError):
    def __init__(self, code: int, what: str):
        super().__init__("cloud_merger_gpu error %d: %s" % (code, what))
        self.code = code


def _outputs(n: int):
    """Host output buffers of a filter for up to n points: (xyzi [n,4] float32, idx [n] uint32)."""
    return np.empty((max(n, 1), 4), np.float32), np.empty(max(n, 1), np.uint32)


def _pack(clouds):
    """Several [n,4] clouds as one float32 array: (array, begin as numpy int64, begin as ctypes int64[], output buffers)."""
    arrs = [np.ascontiguousarray(c, np.float32).reshape(-1, 4) for c in clouds]
    begin = np.concatenate([[0], np.cumsum([len(a) for a in arrs])]).astype(np.int64)
    n = int(begin[-1])
    allpts = np.ascontiguousarray(np.concatenate(arrs)) if n else np.zeros((0, 4), np.float32)
    return allpts, begin, (C.c_int64 * len(begin))(*[int(v) for v in begin]), _outputs(n)


def _part(xyzi, idx, a: int, b: int, base: int = 0):
    """Points [a, b) of host outputs as (xyzi, idx - base): one cloud or zone, its indices relative to its own cloud."""
    return xyzi[a:b].copy(), (idx[a:b].astype(np.int64) - base).astype(np.uint32)


def make_layout(point_step=16, off_x=0, off_y=4, off_z=8, off_intensity=12, is_dense=1) -> CmLayout:
    return CmLayout(point_step, off_x, off_y, off_z, off_intensity, int(is_dense))


@dataclass
class FrameInfo:
    survivor_begin: int
    survivor_end: int
    voxel_begin: int
    voxel_end: int
    min_b: Tuple[int, int, int]
    max_b: Tuple[int, int, int]
    div_b: Tuple[int, int, int]
    pcl_overflow: bool


@dataclass
class FrameResult:
    voxel_xyzi: np.ndarray      # (V, 4) float32 centroids (x, y, z, intensity)
    voxel_count: np.ndarray     # (V,) uint32
    voxel_idx: np.ndarray       # (V,) uint64 PCL voxel index
    survivor_xyzi: np.ndarray   # (M, 4) float32 merged cropped cloud
    survivor_src: np.ndarray    # (M,) uint32 index in the un-cropped concatenation
    info: FrameInfo
    used_mask: int
    stamp: int


def _info(fi: CmFrameInfo) -> FrameInfo:
    return FrameInfo(fi.survivor_begin, fi.survivor_end, fi.voxel_begin, fi.voxel_end, tuple(fi.min_b), tuple(fi.max_b),
                     tuple(fi.div_b), bool(fi.pcl_overflow))


class DeviceBuffer:
    """A device allocation owned through the C ABI (cm_dev_alloc)."""

    def __init__(self, merger: "CloudMerger", nbytes: int):
        self._m = merger
        self.nbytes = int(nbytes)
        p = C.c_void_p()
        merger._check(merger._lib.cm_dev_alloc(merger._h, C.byref(p), C.c_size_t(max(self.nbytes, 16))))
        self.ptr = p.value

    def upload(self, arr: np.ndarray, offset: int = 0) -> "DeviceBuffer":
        a = np.ascontiguousarray(arr)
        assert offset + a.nbytes <= self.nbytes
        self._m._check(self._m._lib.cm_memcpy_h2d(self._m._h, C.c_void_p(self.ptr + offset), a.ctypes.data_as(C.c_void_p),
                                                  C.c_size_t(a.nbytes), None))
        return self

    def free(self):
        if self.ptr:
            self._m._lib.cm_dev_free(self._m._h, C.c_void_p(self.ptr))
            self.ptr = None


class CloudMerger:
    """One handle = one GPU. Mirrors the reference's per-frame flow: submit_cloud() from each sensor callback
    (callbackFrontRight ..., pc_preprocessing_main.cpp:318-508), merge_frame() from the main loop (:574-578)."""

    def __init__(self, device: int = 0, max_sensors: int = 6, max_points_per_sensor: int = 262144,
                 max_point_step: int = 32, frames_in_flight: int = 2, max_batch_points: int = 0,
                 max_batch_frames: int = 1, max_batch_segments: int = 0, out_point_step: int = 16):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        cfg = CmConfig(device, max_sensors, max_points_per_sensor, max_point_step, frames_in_flight, max_batch_points,
                       max_batch_frames, max_batch_segments, out_point_step, 0)
        rc = self._lib.cm_create(C.byref(cfg), C.byref(self._h))
        if rc != _lib.CM_OK:
            self._h = None
            raise CloudMergerError(rc, self._lib.cm_strerror(rc).decode() + " (cm_create; a B200 / sm_100 GPU is required)")
        self.out_point_step = 32 if out_point_step == 32 else 16
        self.max_sensors = max_sensors
        self._buffers: List[DeviceBuffer] = []

    # -- plumbing ----------------------------------------------------------------------------------------------------
    def _check(self, rc: int):
        if rc != _lib.CM_OK:
            raise CloudMergerError(rc, "%s: %s" % (self._lib.cm_strerror(rc).decode(),
                                                   self._lib.cm_last_error(self._h).decode()))

    def close(self):
        if self._h:
            for b in self._buffers:
                b.free()
            self._buffers = []
            self._lib.cm_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- configuration -----------------------------------------------------------------------------------------------
    def set_extrinsic(self, sensor: int, m: np.ndarray, col_major: bool = False):
        """m: 4x4 (or 3x4 / 12 floats row-major) sensor -> base transform (tf::Transform of the reference callbacks)."""
        a = np.asarray(m, np.float32).reshape(-1)
        if a.size == 12:
            a = np.concatenate([a, np.array([0, 0, 0, 1], np.float32)])
        a = np.ascontiguousarray(a[:16])
        self._check(self._lib.cm_set_extrinsic(self._h, sensor, a.ctypes.data_as(C.POINTER(C.c_float)), int(col_major)))

    def set_extrinsic_tf(self, sensor: int, quat_xyzw: Sequence[float], origin_xyz: Sequence[float]):
        q = (C.c_double * 4)(*[float(v) for v in quat_xyzw])
        t = (C.c_double * 3)(*[float(v) for v in origin_xyz])
        self._check(self._lib.cm_set_extrinsic_tf(self._h, sensor, q, t))

    def get_extrinsic(self, sensor: int) -> np.ndarray:
        m = np.empty(12, np.float32)
        self._check(self._lib.cm_get_extrinsic(self._h, sensor, m.ctypes.data_as(C.POINTER(C.c_float))))
        return m

    def set_crop(self, passes: Iterable[Tuple[int, float, float, int]]):
        """passes: (axis, lo, hi, negative) per pcl::PassThrough stage; [] disables cropping."""
        passes = list(passes)
        arr = (CmPass * max(len(passes), 1))()
        for i, (axis, lo, hi, neg) in enumerate(passes):
            arr[i] = CmPass(int(axis), float(np.float32(lo)), float(np.float32(hi)), int(neg))
        self._check(self._lib.cm_set_crop(self._h, len(passes), arr))

    def set_crop_boxes(self, boxes: Sequence[CmCropBox]):
        """pcl::CropBox stages after the PassThrough chain, in order (<= 8; see make_crop_box); [] switches them off. The
        usual one removes the vehicle's own body: make_crop_box(lo, hi, negative=True)."""
        boxes = list(boxes)
        arr = (CmCropBox * max(len(boxes), 1))(*boxes)
        self._check(self._lib.cm_set_crop_boxes(self._h, len(boxes), arr))

    # -- zone slicing: getCloudPart x5 + the z windows of removeGround in one pass (pc_preprocessing_main.cpp:49-92, 228-312)
    def set_zones(self, zones: Sequence[Sequence[Tuple[int, float, float, int]]]):
        """zones: one PassThrough chain [(axis, lo, hi, negative), ...] per zone (<= 16 zones of <= 4 stages)."""
        zones = [list(z) for z in zones]
        arr = (CmZone * max(len(zones), 1))()
        for zi, chain in enumerate(zones):
            if len(chain) > CM_MAX_ZONE_PASSES:
                raise ValueError("a zone takes at most %d stages" % CM_MAX_ZONE_PASSES)
            arr[zi].n_pass = len(chain)
            for k, (axis, lo, hi, neg) in enumerate(chain):
                arr[zi].pass_[k] = CmPass(int(axis), float(np.float32(lo)), float(np.float32(hi)), int(neg))
        self._check(self._lib.cm_set_zones(self._h, len(zones), arr))
        self._n_zones = len(zones)

    def dev_zone_split(self, xyzi_ptr: int = 0, n_points: int = 0, stream: int = 0):
        """Device form; xyzi_ptr = 0 splits the merged cropped cloud of the last transform_crop / run_batch."""
        self._check(self._lib.cm_dev_zone_split(self._h, C.c_void_p(xyzi_ptr or None), C.c_int64(n_points),
                                                C.c_void_p(stream or None)))

    def zone_out(self):
        """(list of (xyzi [n,4] float32, src [n] uint32) per zone) of the last device zone split, downloaded."""
        zo = CmZoneOut()
        self._check(self._lib.cm_get_zone_out(self._h, C.byref(zo)))
        total = int(zo.begin[zo.n_zones])
        xyzi = self.download(zo.xyzi, np.float32, total * 4).reshape(-1, 4) if total else np.zeros((0, 4), np.float32)
        src = self.download(zo.src, np.uint32, total) if total else np.zeros(0, np.uint32)
        return [(xyzi[zo.begin[z]:zo.begin[z + 1]], src[zo.begin[z]:zo.begin[z + 1]]) for z in range(zo.n_zones)]

    def zone_split(self, xyzi: np.ndarray, capacity: Optional[int] = None):
        """Host-buffer form: returns the same per-zone list for a [n,4] float32 cloud in host memory."""
        a = np.ascontiguousarray(xyzi, np.float32).reshape(-1, 4)
        n = len(a)
        cap = int(capacity if capacity is not None else 2 * max(n, 1))
        ox, osrc = _outputs(cap)
        begin = (C.c_int64 * (CM_MAX_ZONES + 1))()
        self._check(self._lib.cm_zone_split(self._h, a.ctypes.data_as(C.c_void_p), C.c_int64(n),
                                            ox.ctypes.data_as(C.c_void_p), osrc.ctypes.data_as(C.c_void_p),
                                            C.c_int64(cap), begin))
        nz = self._n_zones
        return [_part(ox, osrc, begin[z], begin[z + 1]) for z in range(nz)]

    # -- radius outlier removal: outlierRemoval() of the reference (pc_preprocessing_main.cpp:184-192) ----------------------
    def dev_radius_outlier(self, xyzi_ptr: int, n_points: int, radius: float, min_neighbors: int = 1,
                           negative: bool = False, stream: int = 0):
        """Device form; fetch the survivors with radius_outlier_out()."""
        self._check(self._lib.cm_dev_radius_outlier(self._h, C.c_void_p(xyzi_ptr or None), C.c_int64(n_points),
                                                    C.c_double(radius), int(min_neighbors), int(negative),
                                                    C.c_void_p(stream or None)))

    def radius_outlier_out(self):
        """(xyzi [k,4], idx [k]) of the last device radius outlier removal."""
        return self.zone_out()[0]

    def radius_outlier(self, xyzi: np.ndarray, radius: float, min_neighbors: int = 1, negative: bool = False):
        """Host-buffer form: (xyzi [k,4] float32, idx [k] uint32 indices into the input, ascending)."""
        a = np.ascontiguousarray(xyzi, np.float32).reshape(-1, 4)
        n = len(a)
        ox, oi = _outputs(n)
        k = C.c_int64()
        self._check(self._lib.cm_radius_outlier(self._h, a.ctypes.data_as(C.c_void_p), C.c_int64(n), C.c_double(radius),
                                                int(min_neighbors), int(negative), ox.ctypes.data_as(C.c_void_p),
                                                oi.ctypes.data_as(C.c_void_p), C.c_int64(n), C.byref(k)))
        return _part(ox, oi, 0, k.value)

    def dev_radius_outlier_multi(self, xyzi_ptr: int, begin, radius: float, min_neighbors: int = 1, negative: bool = False,
                                 stream: int = 0):
        """Independent clouds [begin[k], begin[k+1]) of one device array in one pass; zone k of zone_out() = survivors of
        cloud k (needs max_batch_frames >= number of clouds)."""
        b = (C.c_int64 * len(begin))(*[int(v) for v in begin])
        self._check(self._lib.cm_dev_radius_outlier_multi(self._h, C.c_void_p(xyzi_ptr or None), b, len(begin) - 1,
                                                          C.c_double(radius), int(min_neighbors), int(negative),
                                                          C.c_void_p(stream or None)))

    def radius_outlier_multi(self, clouds, radius: float, min_neighbors: int = 1, negative: bool = False) -> list:
        """Host-buffer form: per cloud (xyzi [k,4], idx [k] into that cloud)."""
        allpts, begin, b, (ox, oi) = _pack(clouds)
        k, n = len(begin) - 1, len(allpts)
        ob = (C.c_int64 * (k + 1))()
        self._check(self._lib.cm_radius_outlier_multi(self._h, allpts.ctypes.data_as(C.c_void_p), b, k, C.c_double(radius),
                                                      int(min_neighbors), int(negative), ox.ctypes.data_as(C.c_void_p),
                                                      oi.ctypes.data_as(C.c_void_p), C.c_int64(n), ob))
        return [_part(ox, oi, ob[c], ob[c + 1], begin[c]) for c in range(k)]

    # -- statistical outlier removal (pcl::StatisticalOutlierRemoval) --------------------------------------------------------
    @staticmethod
    def _sor_cfg(mean_k, std_mul, negative, sqrt_mode):
        return _lib.CmSorCfg(int(mean_k), int(bool(negative)), int(sqrt_mode), 0, float(std_mul))

    def dev_statistical_outlier(self, xyzi_ptr: int, n_points: int, mean_k: int, std_mul: float, negative: bool = False,
                                sqrt_mode: int = 0, stream: int = 0):
        """Device form; fetch the survivors with radius_outlier_out() / zone_out() and the per-point mean distances and
        per-cloud statistics with statistical_outlier_out()."""
        cfg = self._sor_cfg(mean_k, std_mul, negative, sqrt_mode)
        self._check(self._lib.cm_dev_statistical_outlier(self._h, C.c_void_p(xyzi_ptr or None), C.c_int64(n_points),
                                                         C.byref(cfg), C.c_void_p(stream or None)))

    def dev_statistical_outlier_multi(self, xyzi_ptr: int, begin, mean_k: int, std_mul: float, negative: bool = False,
                                      sqrt_mode: int = 0, stream: int = 0):
        """Independent clouds [begin[k], begin[k+1]) of one device array in one pass; zone k of zone_out() = survivors of
        cloud k (needs max_batch_frames >= number of clouds)."""
        b = (C.c_int64 * len(begin))(*[int(v) for v in begin])
        cfg = self._sor_cfg(mean_k, std_mul, negative, sqrt_mode)
        self._check(self._lib.cm_dev_statistical_outlier_multi(self._h, C.c_void_p(xyzi_ptr or None), b, len(begin) - 1,
                                                               C.byref(cfg), C.c_void_p(stream or None)))

    def statistical_outlier_out(self) -> dict:
        """Of the last statistical outlier removal: "distances" (float32 [n], input order) and "clouds", one dict per cloud
        (mean, stddev, threshold, n_valid, too_few, sum_path), plus "knn_ms" / "sums_ms" (-1 unless profiling)."""
        so = _lib.CmSorOut()
        self._check(self._lib.cm_get_statistical_out(self._h, C.byref(so)))
        n = int(so.n_points)
        dist = self.download(so.distances, np.float32, n) if n else np.zeros(0, np.float32)
        clouds = [{"mean": c.mean, "stddev": c.stddev, "threshold": c.threshold, "n_valid": int(c.n_valid),
                   "too_few": bool(c.too_few), "sum_path": int(c.sum_path)} for c in so.cloud[:so.n_clouds]]
        return {"distances": dist, "clouds": clouds, "knn_ms": float(so.knn_ms), "sums_ms": float(so.sums_ms)}

    def statistical_outlier(self, xyzi: np.ndarray, mean_k: int, std_mul: float, negative: bool = False, sqrt_mode: int = 0):
        """Host-buffer form: (xyzi [k,4] float32, idx [k] uint32 indices into the input, ascending)."""
        a = np.ascontiguousarray(xyzi, np.float32).reshape(-1, 4)
        n = len(a)
        ox, oi = _outputs(n)
        k = C.c_int64()
        cfg = self._sor_cfg(mean_k, std_mul, negative, sqrt_mode)
        self._check(self._lib.cm_statistical_outlier(self._h, a.ctypes.data_as(C.c_void_p), C.c_int64(n), C.byref(cfg),
                                                     ox.ctypes.data_as(C.c_void_p), oi.ctypes.data_as(C.c_void_p),
                                                     C.c_int64(n), C.byref(k)))
        return _part(ox, oi, 0, k.value)

    def statistical_outlier_multi(self, clouds, mean_k: int, std_mul: float, negative: bool = False,
                                  sqrt_mode: int = 0) -> list:
        """Host-buffer form: per cloud (xyzi [k,4], idx [k] into that cloud)."""
        allpts, begin, b, (ox, oi) = _pack(clouds)
        k, n = len(begin) - 1, len(allpts)
        ob = (C.c_int64 * (k + 1))()
        cfg = self._sor_cfg(mean_k, std_mul, negative, sqrt_mode)
        self._check(self._lib.cm_statistical_outlier_multi(self._h, allpts.ctypes.data_as(C.c_void_p), b, k, C.byref(cfg),
                                                           ox.ctypes.data_as(C.c_void_p), oi.ctypes.data_as(C.c_void_p),
                                                           C.c_int64(n), ob))
        return [_part(ox, oi, ob[c], ob[c + 1], begin[c]) for c in range(k)]

    # -- RANSAC ground plane (pcl::SACSegmentation of removeGround, pc_preprocessing_main.cpp:95-117) ------------------------
    @staticmethod
    def _plane_cfg(distance_threshold, probability, max_iterations, optimize, seed, sum_order):
        return _lib.CmPlaneCfg(float(distance_threshold), float(probability), int(max_iterations), int(bool(optimize)),
                               int(seed), int(sum_order))

    @staticmethod
    def _plane_dict(pl) -> dict:
        return {"found": bool(pl.found), "iterations": int(pl.iterations), "draws": int(pl.draws),
                "best_count": int(pl.best_count), "sample": np.array(pl.sample, np.int32),
                "coeff_ransac": np.array(pl.coeff_ransac, np.float32), "coeff": np.array(pl.coeff, np.float32),
                "n_inliers": int(pl.n_inliers)}

    def dev_plane_ransac(self, xyzi_ptr: int, n_points: int, distance_threshold: float, probability: float = 0.99,
                         max_iterations: int = 1000, optimize: bool = True, seed: int = 12345, sum_order: int = 0,
                         stream: int = 0) -> dict:
        """Device form; the ground / no-ground clouds are zones 0 / 1 of zone_out()."""
        cfg = self._plane_cfg(distance_threshold, probability, max_iterations, optimize, seed, sum_order)
        pl = _lib.CmPlane()
        self._check(self._lib.cm_dev_plane_ransac(self._h, C.c_void_p(xyzi_ptr or None), C.c_int64(n_points), C.byref(cfg),
                                                  C.byref(pl), C.c_void_p(stream or None)))
        return self._plane_dict(pl)

    def dev_plane_ransac_multi(self, xyzi_ptr: int, begin, distance_threshold: float, probability: float = 0.99,
                               max_iterations: int = 1000, optimize: bool = True, seed: int = 12345, sum_order: int = 0,
                               stream: int = 0) -> list:
        """Independent plane searches over the consecutive clouds [begin[k], begin[k+1]) of one device array in one pass;
        zone_out() then holds zone 2k = inliers of cloud k, zone 2k + 1 = its other points."""
        b = (C.c_int64 * len(begin))(*[int(v) for v in begin])
        k = len(begin) - 1
        cfg = self._plane_cfg(distance_threshold, probability, max_iterations, optimize, seed, sum_order)
        pl = (_lib.CmPlane * max(k, 1))()
        self._check(self._lib.cm_dev_plane_ransac_multi(self._h, C.c_void_p(xyzi_ptr or None), b, k, C.byref(cfg), pl,
                                                        C.c_void_p(stream or None)))
        return [self._plane_dict(pl[i]) for i in range(k)]

    def plane_ransac_multi(self, clouds, distance_threshold: float, probability: float = 0.99, max_iterations: int = 1000,
                           optimize: bool = True, seed: int = 12345, sum_order: int = 0) -> list:
        """Host-buffer form of dev_plane_ransac_multi: one dict per cloud with "ground" / "rest" as in plane_ransac
        (indices relative to the cloud)."""
        allpts, begin, b, (ox, oi) = _pack(clouds)
        k, n = len(begin) - 1, len(allpts)
        cfg = self._plane_cfg(distance_threshold, probability, max_iterations, optimize, seed, sum_order)
        pl = (_lib.CmPlane * max(k, 1))()
        ob = (C.c_int64 * (2 * k + 1))()
        self._check(self._lib.cm_plane_ransac_multi(self._h, allpts.ctypes.data_as(C.c_void_p), b, k, C.byref(cfg), pl,
                                                    ox.ctypes.data_as(C.c_void_p), oi.ctypes.data_as(C.c_void_p), C.c_int64(n), ob))
        res = []
        for c in range(k):
            r = self._plane_dict(pl[c])
            r["ground"] = _part(ox, oi, ob[2 * c], ob[2 * c + 1], begin[c])
            r["rest"] = _part(ox, oi, ob[2 * c + 1], ob[2 * c + 2], begin[c])
            res.append(r)
        return res

    def plane_ransac(self, xyzi: np.ndarray, distance_threshold: float, probability: float = 0.99,
                     max_iterations: int = 1000, optimize: bool = True, seed: int = 12345, sum_order: int = 0) -> dict:
        """Host-buffer form. Adds "ground" and "rest": (xyzi [k,4] float32, idx [k] uint32 into the input, ascending)."""
        a = np.ascontiguousarray(xyzi, np.float32).reshape(-1, 4)
        n = len(a)
        cfg = self._plane_cfg(distance_threshold, probability, max_iterations, optimize, seed, sum_order)
        pl = _lib.CmPlane()
        ox, oi = _outputs(n)
        begin = (C.c_int64 * 3)()
        self._check(self._lib.cm_plane_ransac(self._h, a.ctypes.data_as(C.c_void_p), C.c_int64(n), C.byref(cfg), C.byref(pl),
                                              ox.ctypes.data_as(C.c_void_p), oi.ctypes.data_as(C.c_void_p), C.c_int64(n),
                                              begin))
        r = self._plane_dict(pl)
        r["ground"], r["rest"] = _part(ox, oi, begin[0], begin[1]), _part(ox, oi, begin[1], begin[2])
        return r

    # -- the body of a proceedX in one call (pc_preprocessing_main.cpp:228-312, :428-446, :474-497) ---------------------------
    def _proceed_cfg(self, parts, roi_z_max, radius, min_neighbors, distance_threshold, probability, max_iterations, optimize,
                     seed, sum_order):
        """parts: (length, deviation, z_max_ground) for a ground-removal part, (length, deviation, None) for a plain one."""
        cfg = _lib.CmProceedCfg()
        cfg.n_parts = len(parts)
        cfg.min_neighbors = int(min_neighbors)
        for k, pt in enumerate(parts):
            zg = pt[2] if len(pt) > 2 else None
            cfg.part[k] = _lib.CmProceedPart(float(np.float32(pt[0])), float(np.float32(pt[1])),
                                             float(np.float32(0.0 if zg is None else zg)), 0 if zg is None else 1)
        cfg.roi_z_max = float(np.float32(roi_z_max))
        cfg.radius = float(radius)
        cfg.plane = self._plane_cfg(distance_threshold, probability, max_iterations, optimize, seed, sum_order)
        return cfg

    def dev_proceed_zones(self, roi_ptr: int, n_points: int, parts, roi_z_max: float = 3.0, radius: float = 0.15,
                          min_neighbors: int = 1, distance_threshold: float = 0.3, probability: float = 0.99,
                          max_iterations: int = 1000, optimize: bool = True, seed: int = 12345, sum_order: int = 0,
                          stream: int = 0) -> dict:
        """Device form: the ROI cloud at roi_ptr -> no-ground / ground clouds in device memory (pointers + sizes)."""
        cfg = self._proceed_cfg(parts, roi_z_max, radius, min_neighbors, distance_threshold, probability, max_iterations,
                                optimize, seed, sum_order)
        po = _lib.CmProceedOut()
        self._check(self._lib.cm_dev_proceed_zones(self._h, C.c_void_p(roi_ptr or None), C.c_int64(n_points), C.byref(cfg),
                                                   C.byref(po), C.c_void_p(stream or None)))
        return {"no_ground_ptr": po.no_ground_xyzi, "n_no_ground": int(po.n_no_ground), "ground_ptr": po.ground_xyzi,
                "n_ground": int(po.n_ground), "planes": [self._plane_dict(po.plane[i]) for i in range(po.n_planes)],
                "host_syncs": int(po.host_syncs)}

    def proceed_zones(self, roi_xyzi: np.ndarray, parts, roi_z_max: float = 3.0, radius: float = 0.15, min_neighbors: int = 1,
                      distance_threshold: float = 0.3, probability: float = 0.99, max_iterations: int = 1000,
                      optimize: bool = True, seed: int = 12345, sum_order: int = 0) -> dict:
        """Host-buffer form: (no_ground [n,4], ground [m,4], planes)."""
        a = np.ascontiguousarray(roi_xyzi, np.float32).reshape(-1, 4)
        n = len(a)
        cfg = self._proceed_cfg(parts, roi_z_max, radius, min_neighbors, distance_threshold, probability, max_iterations,
                                optimize, seed, sum_order)
        cap = 2 * max(n, 1)
        ng, g = np.empty((cap, 4), np.float32), np.empty((cap, 4), np.float32)
        n_ng, n_g = C.c_int64(), C.c_int64()
        pl = (_lib.CmPlane * _lib.CM_MAX_PROCEED_PARTS)()
        self._check(self._lib.cm_proceed_zones(self._h, a.ctypes.data_as(C.c_void_p), C.c_int64(n), C.byref(cfg),
                                               ng.ctypes.data_as(C.c_void_p), C.c_int64(cap), C.byref(n_ng),
                                               g.ctypes.data_as(C.c_void_p), C.c_int64(cap), C.byref(n_g), pl))
        k = sum(1 for pt in parts if len(pt) > 2 and pt[2] is not None)
        return {"no_ground": ng[:n_ng.value].copy(), "ground": g[:n_g.value].copy(),
                "planes": [self._plane_dict(pl[i]) for i in range(k)]}

    # -- giant-cloud mode: device-side pieces of the voxel-key range partition (BASELINE config 4) -------------------------
    def dev_bounds(self, xyzi_ptr: int, n_points: int, stream: int = 0):
        """pcl::getMinMax3D of n packed points on the device -> (min[3], max[3] float32, number of finite points)."""
        mn, mx = (C.c_float * 3)(), (C.c_float * 3)()
        nf = C.c_int64()
        self._check(self._lib.cm_dev_bounds(self._h, C.c_void_p(xyzi_ptr or None), C.c_int64(n_points), mn, mx,
                                            C.byref(nf), C.c_void_p(stream or None)))
        return np.array(mn, np.float32), np.array(mx, np.float32), nf.value

    def dev_key_histogram(self, xyzi_ptr: int, n_points: int, min_p, max_p, bins: int, hist_ptr: int, stream: int = 0) -> int:
        """Histogram of the PCL voxel index on the grid of the box [min_p, max_p] into `bins` uint64 device counters;
        returns the key width of a bin."""
        mn = (C.c_float * 3)(*[float(v) for v in min_p]); mx = (C.c_float * 3)(*[float(v) for v in max_p])
        width = C.c_uint64()
        self._check(self._lib.cm_dev_key_histogram(self._h, C.c_void_p(xyzi_ptr or None), C.c_int64(n_points), mn, mx,
                                                   int(bins), C.c_void_p(hist_ptr), C.byref(width), C.c_void_p(stream or None)))
        return int(width.value)

    def dev_route_by_key(self, xyzi_ptr: int, n_points: int, min_p, max_p, splitters, invalid_part: int, stream: int = 0):
        """Groups the points by key range (len(splitters) + 1 parts); fetch the device arrays with zone_out_raw()."""
        mn = (C.c_float * 3)(*[float(v) for v in min_p]); mx = (C.c_float * 3)(*[float(v) for v in max_p])
        sp = [int(v) for v in splitters]
        arr = (C.c_uint64 * max(len(sp), 1))(*sp)
        self._check(self._lib.cm_dev_route_by_key(self._h, C.c_void_p(xyzi_ptr or None), C.c_int64(n_points), mn, mx, arr,
                                                  len(sp) + 1, int(invalid_part), C.c_void_p(stream or None)))

    def zone_out_raw(self):
        """(device pointer of the grouped xyzi, device pointer of the source indices, begin offsets) of the last split."""
        zo = CmZoneOut()
        self._check(self._lib.cm_get_zone_out(self._h, C.byref(zo)))
        return zo.xyzi, zo.src, [int(zo.begin[k]) for k in range(zo.n_zones + 1)]

    def stream_create(self) -> int:
        p = C.c_void_p()
        self._check(self._lib.cm_stream_create(self._h, C.byref(p)))
        return int(p.value)

    def stream_destroy(self, stream: int):
        self._check(self._lib.cm_stream_destroy(self._h, C.c_void_p(stream or None)))

    def stream_sync(self, stream: int):
        self._check(self._lib.cm_stream_sync(self._h, C.c_void_p(stream or None)))

    def memcpy_d2d(self, dst_ptr: int, src_ptr: int, nbytes: int, stream: int = 0):
        self._check(self._lib.cm_memcpy_d2d(self._h, C.c_void_p(dst_ptr), C.c_void_p(src_ptr), C.c_size_t(nbytes),
                                            C.c_void_p(stream or None)))

    def set_voxel(self, leaf, min_points: int = 2, downsample_all: bool = True):
        leaf = np.broadcast_to(np.asarray(leaf, np.float32), (3,)).copy()
        self._check(self._lib.cm_set_voxel(self._h, leaf.ctypes.data_as(C.POINTER(C.c_float)), int(min_points),
                                           int(downsample_all)))

    def set_voxel_bounds(self, min3=None, max3=None):
        """Bounding box of the whole (partitioned) cloud for the next dev_voxelgrid calls; None switches it off."""
        if min3 is None or max3 is None:
            self._check(self._lib.cm_set_voxel_bounds(self._h, None, None))
            return
        a = (C.c_float * 3)(*[float(np.float32(v)) for v in min3])
        b = (C.c_float * 3)(*[float(np.float32(v)) for v in max3])
        self._check(self._lib.cm_set_voxel_bounds(self._h, a, b))

    def set_overflow_mode(self, pcl_like: bool):
        self._check(self._lib.cm_set_overflow_mode(self._h, int(pcl_like)))

    def set_submit_policy(self, first_wins: bool):
        """False (default): the newest cloud of a sensor is merged (my_cloud_fusion); True: the first one after the previous
        merge, later ones are dropped -- pcl_preprocessing's flag gate (pc_preprocessing_main.cpp:330)."""
        self._check(self._lib.cm_set_submit_policy(self._h, 1 if first_wins else 0))

    def set_profiling(self, on: bool):
        self._check(self._lib.cm_set_profiling(self._h, int(on)))

    # -- host path ---------------------------------------------------------------------------------------------------
    def submit_cloud(self, sensor: int, data, n_points: int, layout: CmLayout, stamp: int = 0, pinned: bool = False):
        """data: numpy buffer (any dtype) holding n_points records of layout.point_step bytes, or a raw address."""
        if isinstance(data, int):
            ptr = C.c_void_p(data)
        else:
            a = np.ascontiguousarray(data)
            assert a.nbytes >= n_points * layout.point_step
            ptr = a.ctypes.data_as(C.c_void_p)
        fn = self._lib.cm_submit_cloud_pinned if pinned else self._lib.cm_submit_cloud
        self._check(fn(self._h, sensor, ptr, n_points, C.byref(layout), C.c_uint64(stamp)))

    def submit_clouds_pinned(self, sensors: Sequence[int], addresses: Sequence[int], n_points: Sequence[int],
                             layouts: Sequence[CmLayout], stamps: Optional[Sequence[int]] = None):
        """All page-locked clouds of a frame in one call (cm_submit_clouds_pinned): host-adjacent clouds of consecutive
        sensors go over PCIe as one copy. addresses are raw host addresses."""
        k = len(sensors)
        a_s = (C.c_int * k)(*[int(x) for x in sensors])
        a_d = (C.c_void_p * k)(*[int(x) for x in addresses])
        a_n = (C.c_int64 * k)(*[int(x) for x in n_points])
        a_l = (CmLayout * k)(*layouts)
        a_t = (C.c_uint64 * k)(*[int(x) for x in (stamps if stamps is not None else [0] * k)])
        self._check(self._lib.cm_submit_clouds_pinned(self._h, k, a_s, a_d, a_n, a_l, a_t))

    def prepared_frame_submit(self, sensors, addresses, n_points, layouts, stamp: int = 0):
        """The argument arrays of submit_clouds_pinned built once, for callers that replay the same buffers every frame;
        returns a zero-argument callable."""
        k = len(sensors)
        a_s = (C.c_int * k)(*[int(x) for x in sensors])
        a_d = (C.c_void_p * k)(*[int(x) for x in addresses])
        a_n = (C.c_int64 * k)(*[int(x) for x in n_points])
        a_l = (CmLayout * k)(*layouts)
        a_t = (C.c_uint64 * k)(*([int(stamp)] * k))
        fn, h, chk = self._lib.cm_submit_clouds_pinned, self._h, self._check

        def go():
            chk(fn(h, k, a_s, a_d, a_n, a_l, a_t))
        return go

    def merge_frame_async(self, sensor_mask: int = (1 << 64) - 1) -> int:
        t = C.c_int64()
        self._check(self._lib.cm_merge_frame_async(self._h, C.c_uint64(sensor_mask), C.byref(t)))
        return t.value

    def _make_out(self, voxel_cap: int, surv_cap: int, want_survivors: bool):
        step_f = self.out_point_step // 4
        bufs = dict(vx=np.empty((max(voxel_cap, 1), step_f), np.float32), vc=np.empty(max(voxel_cap, 1), np.uint32),
                    vi=np.empty(max(voxel_cap, 1), np.uint64))
        out = CmFrameOut()
        out.voxel_xyzi = bufs["vx"].ctypes.data
        out.voxel_capacity = voxel_cap
        out.voxel_count = bufs["vc"].ctypes.data
        out.voxel_idx = bufs["vi"].ctypes.data
        if want_survivors:
            bufs["sx"] = np.empty((max(surv_cap, 1), 4), np.float32)
            bufs["ss"] = np.empty(max(surv_cap, 1), np.uint32)
            out.survivor_xyzi = bufs["sx"].ctypes.data
            out.survivor_src = bufs["ss"].ctypes.data
            out.survivor_capacity = surv_cap
        return out, bufs

    def _result(self, out: CmFrameOut, bufs, used: int, stamp: int) -> FrameResult:
        v, m = out.n_voxels, out.n_survivors
        vx = bufs["vx"][:v]
        if self.out_point_step == 32:
            vx = np.concatenate([vx[:, 0:3], vx[:, 4:5]], axis=1)
        sx = bufs["sx"][:m].copy() if "sx" in bufs else np.zeros((0, 4), np.float32)
        ss = bufs["ss"][:m].copy() if "ss" in bufs else np.zeros(0, np.uint32)
        res = FrameResult(vx.copy(), bufs["vc"][:v].copy(), bufs["vi"][:v].copy(), sx, ss, _info(out.info), used, stamp)
        res.raw_voxel_records = bufs["vx"][:v].copy()
        return res

    def make_frame_buffers(self, capacity: int, want_survivors: bool = False, pinned: bool = True):
        """Reusable (page-locked) result buffers for wait_frame_into(): no per-frame allocation on the hot path."""
        step = self.out_point_step

        def alloc(nbytes, dtype, shape):
            if pinned:
                raw, _ = host_alloc(nbytes)
                return raw.view(dtype).reshape(shape)
            return np.empty(shape, dtype)
        cap = max(capacity, 1)
        bufs = dict(vx=alloc(cap * step, np.float32, (cap, step // 4)), vc=alloc(cap * 4, np.uint32, (cap,)),
                    vi=alloc(cap * 8, np.uint64, (cap,)))
        out = CmFrameOut()
        out.voxel_xyzi = bufs["vx"].ctypes.data
        out.voxel_capacity = capacity
        out.voxel_count = bufs["vc"].ctypes.data
        out.voxel_idx = bufs["vi"].ctypes.data
        if want_survivors:
            bufs["sx"] = alloc(cap * 16, np.float32, (cap, 4))
            bufs["ss"] = alloc(cap * 4, np.uint32, (cap,))
            out.survivor_xyzi = bufs["sx"].ctypes.data
            out.survivor_src = bufs["ss"].ctypes.data
            out.survivor_capacity = capacity
        return out, bufs

    def wait_frame_into(self, ticket: int, out: CmFrameOut) -> CmFrameOut:
        """cm_wait_frame into caller-owned buffers (see make_frame_buffers); returns `out` with the counts filled in."""
        self._check(self._lib.cm_wait_frame(self._h, ticket, C.byref(out), None, None))
        return out

    def wait_frame_view(self, ticket: int, view: Optional["_lib.CmFrameView"] = None):
        """cm_wait_frame_view: one synchronisation, no copy -- the returned struct points into the library's page-locked
        result mirrors of that frame (valid until frames_in_flight further frames have been merged). view_arrays() wraps
        them as numpy arrays without copying."""
        v = view if view is not None else _lib.CmFrameView()
        self._check(self._lib.cm_wait_frame_view(self._h, ticket, C.byref(v)))
        return v

    def view_arrays(self, v) -> dict:
        n, step_f = int(v.n_voxels), self.out_point_step // 4
        if n == 0:
            return dict(voxel_xyzi=np.zeros((0, step_f), np.float32), voxel_count=np.zeros(0, np.uint32), voxel_idx=np.zeros(0, np.uint64))

        def arr(ptr, dtype, count):
            return np.frombuffer((C.c_uint8 * (count * np.dtype(dtype).itemsize)).from_address(ptr), dtype=dtype, count=count)
        return dict(voxel_xyzi=arr(v.voxel_xyzi, np.float32, n * step_f).reshape(n, step_f), voxel_count=arr(v.voxel_count, np.uint32, n),
                    voxel_idx=arr(v.voxel_idx, np.uint64, n))

    def wait_frame(self, ticket: int, capacity: int, want_survivors: bool = True) -> FrameResult:
        out, bufs = self._make_out(capacity, capacity, want_survivors)
        used, stamp = C.c_uint64(), C.c_uint64()
        self._check(self._lib.cm_wait_frame(self._h, ticket, C.byref(out), C.byref(used), C.byref(stamp)))
        return self._result(out, bufs, used.value, stamp.value)

    def merge_frame(self, capacity: int, sensor_mask: int = (1 << 64) - 1, want_survivors: bool = True) -> FrameResult:
        """fusePointclouds + voxelgrid of the reference main loop (pc_preprocessing_main.cpp:574-578)."""
        out, bufs = self._make_out(capacity, capacity, want_survivors)
        used, stamp = C.c_uint64(), C.c_uint64()
        self._check(self._lib.cm_merge_frame(self._h, C.c_uint64(sensor_mask), C.byref(out), C.byref(used),
                                             C.byref(stamp)))
        return self._result(out, bufs, used.value, stamp.value)

    # -- device path -------------------------------------------------------------------------------------------------
    def device_buffer(self, nbytes: int) -> DeviceBuffer:
        b = DeviceBuffer(self, nbytes)
        self._buffers.append(b)
        return b

    def upload(self, arr: np.ndarray) -> DeviceBuffer:
        a = np.ascontiguousarray(arr)
        b = self.device_buffer(a.nbytes)
        self._check(self._lib.cm_memcpy_h2d(self._h, C.c_void_p(b.ptr), a.ctypes.data_as(C.c_void_p),
                                            C.c_size_t(a.nbytes), None))
        return b

    def download(self, ptr: int, dtype, count: int) -> np.ndarray:
        out = np.empty(count, dtype)
        if count:
            self._check(self._lib.cm_memcpy_d2h(self._h, out.ctypes.data_as(C.c_void_p), C.c_void_p(ptr),
                                                C.c_size_t(out.nbytes), None))
        return out

    @staticmethod
    def make_segments(items) -> "C.Array":
        """items: iterable of (device_ptr, n_points, CmLayout, sensor, frame)."""
        items = list(items)
        arr = (CmSegment * max(len(items), 1))()
        for i, (ptr, n, layout, sensor, frame) in enumerate(items):
            arr[i].data = ptr
            arr[i].n_points = int(n)
            arr[i].layout = layout
            arr[i].sensor = int(sensor)
            arr[i].frame = int(frame)
        arr._n = len(items)
        return arr

    def run_batch(self, segments, n_segments: Optional[int] = None, stream: int = 0):
        n = n_segments if n_segments is not None else getattr(segments, "_n", len(segments))
        self._check(self._lib.cm_run_batch(self._h, segments, n, C.c_void_p(stream)))

    def dev_transform_crop(self, segments, n_segments: Optional[int] = None, stream: int = 0):
        n = n_segments if n_segments is not None else getattr(segments, "_n", len(segments))
        self._check(self._lib.cm_dev_transform_crop(self._h, segments, n, C.c_void_p(stream)))

    def dev_voxelgrid(self, xyzi_ptr: int, n_points: int, is_dense: bool = True, stream: int = 0):
        self._check(self._lib.cm_dev_voxelgrid(self._h, C.c_void_p(xyzi_ptr), n_points, int(is_dense), C.c_void_p(stream)))

    def sync(self):
        self._check(self._lib.cm_sync(self._h))

    def stats(self) -> CmStats:
        s = CmStats()
        self._check(self._lib.cm_get_stats(self._h, C.byref(s)))
        return s

    def frame_info(self) -> List[FrameInfo]:
        n = C.c_int()
        self._check(self._lib.cm_get_frame_info(self._h, None, 0, C.byref(n)))
        arr = (CmFrameInfo * max(n.value, 1))()
        self._check(self._lib.cm_get_frame_info(self._h, arr, n.value, C.byref(n)))
        return [_info(arr[i]) for i in range(n.value)]

    def device_out(self) -> CmDeviceOut:
        o = CmDeviceOut()
        self._check(self._lib.cm_get_device_out(self._h, C.byref(o)))
        return o

    def launch_count(self) -> int:
        return int(self._lib.cm_launch_count(self._h))

    def stage_ms(self, stage: str) -> float:
        v = C.c_float()
        self._check(self._lib.cm_stage_ms(self._h, stage.encode(), C.byref(v)))
        return v.value

    def fetch_batch_outputs(self, want_sorted: bool = True) -> dict:
        """Downloads everything the last device run produced (test helper; sizes come from the run's stats)."""
        st = self.stats()
        o = self.device_out()
        m, v = int(st.survivors), int(st.voxels_out)
        res = dict(stats=st, frames=self.frame_info(), key_bytes=o.key_bytes, key_idx_bits=o.key_idx_bits)
        res["survivor_xyzi"] = self.download(o.survivor_xyzi, np.float32, m * 4).reshape(m, 4) if o.survivor_xyzi else None
        res["survivor_src"] = self.download(o.survivor_src, np.uint32, m) if o.survivor_src else None
        res["survivor_slot"] = self.download(o.survivor_slot, np.uint32, m) if o.survivor_slot else None
        if o.voxel_xyzi:
            step_f = self.out_point_step // 4
            vx = self.download(o.voxel_xyzi, np.float32, v * step_f).reshape(v, step_f)
            res["voxel_records"] = vx
            res["voxel_xyzi"] = vx if step_f == 4 else np.concatenate([vx[:, 0:3], vx[:, 4:5]], axis=1)
            res["voxel_count"] = self.download(o.voxel_count, np.uint32, v)
            res["voxel_idx"] = self.download(o.voxel_idx, np.uint64, v)
            if want_sorted:
                kd = np.uint32 if o.key_bytes == 4 else np.uint64
                res["sorted_key"] = self.download(o.sorted_key, kd, m).astype(np.uint64)
                slot = self.download(o.sorted_point, np.uint32, m)
                res["sorted_slot"] = slot
                if res["survivor_slot"] is not None and m:   # slot -> dense survivor index
                    inv = np.full(int(res["survivor_slot"].max()) + 1, 0xFFFFFFFF, np.uint32)
                    inv[res["survivor_slot"]] = np.arange(m, dtype=np.uint32)
                    res["sorted_point"] = inv[slot]
                else:
                    res["sorted_point"] = slot
        return res


def giant_unique_id() -> bytes:
    """ncclGetUniqueId through the C ABI (rank 0 calls it and ships the 128 bytes to every rank)."""
    lib = _lib.load()
    buf = C.create_string_buffer(_lib.CM_GIANT_ID_BYTES)
    rc = lib.cm_giant_unique_id(buf)
    if rc != _lib.CM_OK:
        raise CloudMergerError(rc, "cm_giant_unique_id (is libnccl.so.2 loadable?)")
    return buf.raw


class GiantCloud:
    """BASELINE config 4 behind the C ABI (cm_giant_*): VoxelGrid of one cloud block-distributed over the GPUs of a box --
    C++ + NCCL inside the library (bounding-box and histogram all-reduces, device-side splitters, one all-to-all, local
    VoxelGrid). nccl_id=None with world > 1 gives a dry object that stops after the grouping (single-GPU tests)."""

    def __init__(self, merger: CloudMerger, rank: int, world: int, nccl_id: Optional[bytes] = None):
        self.m = merger
        self.rank, self.world = rank, world
        self._g = C.c_void_p()
        idp = C.create_string_buffer(nccl_id, _lib.CM_GIANT_ID_BYTES) if nccl_id is not None else None
        merger._check(merger._lib.cm_giant_create(merger._h, rank, world, idp, C.byref(self._g)))

    def close(self):
        if self._g:
            self.m._lib.cm_giant_destroy(self._g)
            self._g = None

    def voxelgrid(self, xyzi_ptr: int, n_local: int, stream: int = 0) -> dict:
        """Enqueues the whole partitioned VoxelGrid of this rank's block; the voxels are fetched like any other run's
        (merger.stats() / device_out())."""
        info = _lib.CmGiantInfo()
        rc = self.m._lib.cm_giant_voxelgrid(self._g, C.c_void_p(xyzi_ptr or None), C.c_int64(n_local), C.byref(info),
                                            C.c_void_p(stream or None))
        if rc != _lib.CM_OK:
            raise CloudMergerError(rc, self.m._lib.cm_giant_last_error(self._g).decode())
        w = self.world
        return {"points_received": int(info.points_received), "points_sent_away": int(info.points_sent_away),
                "points_total_finite": int(info.points_total_finite), "splitters": [int(info.splitter[r]) for r in range(w - 1)],
                "min_p": np.array(info.min_p, np.float32), "max_p": np.array(info.max_p, np.float32),
                "min_b": np.array(info.min_b, np.int64), "div_b": np.array(info.div_b, np.int64), "key_bits": int(info.key_bits),
                "host_syncs": int(info.host_syncs), "send_begin": [int(info.send_begin[r]) for r in range(w + 1)],
                "exchange": {0: "none", 1: "nccl", 2: "peer"}.get(int(info.exchange), "?"),
                "stage_ms": [float(x) for x in info.stage_ms]}


def host_alloc(nbytes: int) -> Tuple[np.ndarray, int]:
    """Page-locked host memory as a uint8 numpy array (cm_host_alloc). Returns (array, address); never freed by GC."""
    lib = _lib.load()
    p = C.c_void_p()
    rc = lib.cm_host_alloc(C.byref(p), C.c_size_t(max(nbytes, 1)))
    if rc != _lib.CM_OK:
        raise CloudMergerError(rc, "cm_host_alloc(%d)" % nbytes)
    buf = (C.c_uint8 * max(nbytes, 1)).from_address(p.value)
    return np.frombuffer(buf, dtype=np.uint8, count=nbytes), p.value
