"""ctypes binding of libcloud_merger_gpu.so -- the C ABI of include/cloud_merger_gpu.h.

The product path has no CPU fallback: if the shared library is missing or cannot be loaded this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcloud_merger_gpu.so")

CM_OK, CM_E_INVALID, CM_E_CAPACITY, CM_E_CUDA, CM_E_NO_DEVICE, CM_E_KEY_RANGE, CM_E_INTERNAL, CM_E_NOT_READY = range(8)
CM_MAX_PASSES = 8
CM_MAX_SENSORS = 64
CM_NO_FIELD = -1


class CmPass(C.Structure):
    _fields_ = [("axis", C.c_int32), ("lo", C.c_float), ("hi", C.c_float), ("negative", C.c_int32)]


CM_MAX_CROP_BOXES = 8


class CmCropBox(C.Structure):
    _fields_ = [("min", C.c_float * 3), ("max", C.c_float * 3), ("translation", C.c_float * 3), ("rotation", C.c_float * 3),
                ("transform", C.c_float * 12), ("negative", C.c_int32), ("reserved", C.c_int32)]


CM_MAX_ZONES = 16
CM_MAX_ZONE_PASSES = 4


class CmZone(C.Structure):
    _fields_ = [("n_pass", C.c_int32), ("pass_", CmPass * CM_MAX_ZONE_PASSES)]


class CmZoneOut(C.Structure):
    _fields_ = [("xyzi", C.c_void_p), ("src", C.c_void_p), ("begin", C.c_int64 * (CM_MAX_ZONES + 1)),
                ("n_zones", C.c_int32), ("reserved", C.c_int32)]


class CmPlaneCfg(C.Structure):
    _fields_ = [("distance_threshold", C.c_double), ("probability", C.c_double), ("max_iterations", C.c_int32),
                ("optimize", C.c_int32), ("seed", C.c_uint32), ("sum_order", C.c_int32)]


class CmPlane(C.Structure):
    _fields_ = [("found", C.c_int32), ("iterations", C.c_int32), ("draws", C.c_int32), ("best_count", C.c_int32),
                ("sample", C.c_int32 * 3), ("reserved", C.c_int32), ("coeff_ransac", C.c_float * 4),
                ("coeff", C.c_float * 4), ("n_inliers", C.c_int64)]


CM_SUM4_SSE2, CM_SUM4_SSE3, CM_SUM4_SCALAR = 0, 1, 2

CM_SOR_MAX_K = 127
CM_SOR_SQRT_FLOAT, CM_SOR_SQRT_DOUBLE = 0, 1
CM_SOR_SUM_SERIAL, CM_SOR_SQ_SUM_SERIAL = 1, 2


class CmSorCfg(C.Structure):
    _fields_ = [("mean_k", C.c_int32), ("negative", C.c_int32), ("sqrt_mode", C.c_int32), ("reserved", C.c_int32),
                ("std_mul", C.c_double)]


class CmSorStats(C.Structure):
    _fields_ = [("mean", C.c_double), ("stddev", C.c_double), ("threshold", C.c_double), ("n_valid", C.c_int64),
                ("too_few", C.c_int32), ("sum_path", C.c_int32)]


class CmSorOut(C.Structure):
    _fields_ = [("distances", C.c_void_p), ("n_points", C.c_int64), ("n_clouds", C.c_int32), ("reserved", C.c_int32),
                ("knn_ms", C.c_float), ("sums_ms", C.c_float), ("cloud", CmSorStats * CM_MAX_ZONES)]
CM_MAX_PROCEED_PARTS = 8


CM_GIANT_ID_BYTES = 128


class CmGiantInfo(C.Structure):
    _fields_ = [("points_local", C.c_int64), ("points_received", C.c_int64), ("points_sent_away", C.c_int64),
                ("points_total_finite", C.c_int64), ("voxels_local", C.c_int64), ("splitter", C.c_uint64 * CM_MAX_ZONES),
                ("min_p", C.c_float * 3), ("max_p", C.c_float * 3), ("min_b", C.c_int32 * 3), ("div_b", C.c_int32 * 3),
                ("key_bits", C.c_int32), ("host_syncs", C.c_int32), ("exchange", C.c_int32), ("reserved", C.c_int32),
                ("stage_ms", C.c_float * 4),
                ("send_begin", C.c_int64 * (CM_MAX_ZONES + 1))]


class CmProceedPart(C.Structure):
    _fields_ = [("length", C.c_float), ("deviation", C.c_float), ("z_max_ground", C.c_float), ("ground_removal", C.c_int32)]


class CmProceedCfg(C.Structure):
    _fields_ = [("n_parts", C.c_int32), ("min_neighbors", C.c_int32), ("part", CmProceedPart * CM_MAX_PROCEED_PARTS),
                ("roi_z_max", C.c_float), ("reserved", C.c_float), ("radius", C.c_double), ("plane", CmPlaneCfg)]


class CmProceedOut(C.Structure):
    _fields_ = [("no_ground_xyzi", C.c_void_p), ("ground_xyzi", C.c_void_p), ("n_no_ground", C.c_int64),
                ("n_ground", C.c_int64), ("plane", CmPlane * CM_MAX_PROCEED_PARTS), ("n_planes", C.c_int32),
                ("host_syncs", C.c_int32)]


class CmLayout(C.Structure):
    _fields_ = [("point_step", C.c_int32), ("off_x", C.c_int32), ("off_y", C.c_int32), ("off_z", C.c_int32),
                ("off_intensity", C.c_int32), ("is_dense", C.c_int32)]


class CmPc2Field(C.Structure):
    _fields_ = [("name", C.c_char_p), ("offset", C.c_uint32), ("datatype", C.c_uint8), ("count", C.c_uint32)]


class CmPc2Desc(C.Structure):
    _fields_ = [("height", C.c_uint32), ("width", C.c_uint32), ("point_step", C.c_uint32), ("row_step", C.c_uint32),
                ("is_bigendian", C.c_int32), ("is_dense", C.c_int32), ("n_fields", C.c_int32), ("fields", CmPc2Field * 4)]


CM_PC2_FLOAT32 = 7


class CmSegment(C.Structure):
    _fields_ = [("data", C.c_void_p), ("n_points", C.c_int64), ("layout", CmLayout), ("sensor", C.c_int32),
                ("frame", C.c_int32)]


class CmConfig(C.Structure):
    _fields_ = [("device", C.c_int32), ("max_sensors", C.c_int32), ("max_points_per_sensor", C.c_int64),
                ("max_point_step", C.c_int32), ("frames_in_flight", C.c_int32), ("max_batch_points", C.c_int64),
                ("max_batch_frames", C.c_int32), ("max_batch_segments", C.c_int32), ("out_point_step", C.c_int32),
                ("reserved", C.c_int32)]


class CmStats(C.Structure):
    _fields_ = [("points_in", C.c_int64), ("survivors", C.c_int64), ("voxels_out", C.c_int64), ("frames", C.c_int32),
                ("key_bits", C.c_int32), ("sort_passes", C.c_int32), ("key_bytes", C.c_int32),
                ("pcl_overflow", C.c_int32), ("device_error", C.c_int32), ("gpu_ms", C.c_float),
                ("reserved", C.c_float)]


class CmFrameInfo(C.Structure):
    _fields_ = [("survivor_begin", C.c_int64), ("survivor_end", C.c_int64), ("voxel_begin", C.c_int64),
                ("voxel_end", C.c_int64), ("min_b", C.c_int32 * 3), ("max_b", C.c_int32 * 3),
                ("div_b", C.c_int32 * 3), ("pcl_overflow", C.c_int32)]


class CmDeviceOut(C.Structure):
    _fields_ = [("survivor_xyzi", C.c_void_p), ("survivor_src", C.c_void_p), ("survivor_slot", C.c_void_p),
                ("slot_xyzi", C.c_void_p), ("sorted_key", C.c_void_p),
                ("sorted_point", C.c_void_p), ("voxel_xyzi", C.c_void_p), ("voxel_count", C.c_void_p),
                ("voxel_idx", C.c_void_p), ("key_bytes", C.c_int32), ("key_idx_bits", C.c_int32)]


class CmFrameOut(C.Structure):
    _fields_ = [("voxel_xyzi", C.c_void_p), ("voxel_capacity", C.c_int64), ("voxel_count", C.c_void_p),
                ("voxel_idx", C.c_void_p), ("survivor_xyzi", C.c_void_p), ("survivor_capacity", C.c_int64),
                ("survivor_src", C.c_void_p), ("n_voxels", C.c_int64), ("n_survivors", C.c_int64),
                ("info", CmFrameInfo)]


class CmFrameView(C.Structure):
    _fields_ = [("voxel_xyzi", C.c_void_p), ("voxel_count", C.c_void_p), ("voxel_idx", C.c_void_p), ("n_voxels", C.c_int64),
                ("n_survivors", C.c_int64), ("info", CmFrameInfo), ("used_mask", C.c_uint64), ("stamp", C.c_uint64)]


# every symbol include/cloud_merger_gpu.h declares: name -> (restype, argtypes)
_H = C.c_void_p
SYMBOLS = {
    "cm_create": (C.c_int, [C.POINTER(CmConfig), C.POINTER(_H)]),
    "cm_destroy": (C.c_int, [_H]),
    "cm_strerror": (C.c_char_p, [C.c_int]),
    "cm_last_error": (C.c_char_p, [_H]),
    "cm_version": (C.c_char_p, []),
    "cm_device_count": (C.c_int, []),
    "cm_layout_from_pointcloud2": (C.c_int, [C.POINTER(CmPc2Field), C.c_int, C.c_uint32, C.c_int, C.c_int, C.POINTER(CmLayout)]),
    "cm_pointcloud2_describe": (C.c_int, [C.c_int, C.c_int64, C.POINTER(CmPc2Desc)]),
    "cm_set_extrinsic": (C.c_int, [_H, C.c_int, C.POINTER(C.c_float), C.c_int]),
    "cm_set_extrinsic_tf": (C.c_int, [_H, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "cm_get_extrinsic": (C.c_int, [_H, C.c_int, C.POINTER(C.c_float)]),
    "cm_set_crop": (C.c_int, [_H, C.c_int, C.POINTER(CmPass)]),
    "cm_set_crop_boxes": (C.c_int, [_H, C.c_int, C.POINTER(CmCropBox)]),
    "cm_set_voxel": (C.c_int, [_H, C.POINTER(C.c_float), C.c_int, C.c_int]),
    "cm_set_voxel_bounds": (C.c_int, [_H, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "cm_set_overflow_mode": (C.c_int, [_H, C.c_int]),
    "cm_set_submit_policy": (C.c_int, [_H, C.c_int]),
    "cm_submit_cloud": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int64, C.POINTER(CmLayout), C.c_uint64]),
    "cm_submit_cloud_pinned": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int64, C.POINTER(CmLayout), C.c_uint64]),
    "cm_submit_clouds_pinned": (C.c_int, [_H, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                          C.POINTER(CmLayout), C.POINTER(C.c_uint64)]),
    "cm_merge_frame": (C.c_int, [_H, C.c_uint64, C.POINTER(CmFrameOut), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "cm_merge_frame_async": (C.c_int, [_H, C.c_uint64, C.POINTER(C.c_int64)]),
    "cm_wait_frame": (C.c_int, [_H, C.c_int64, C.POINTER(CmFrameOut), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "cm_wait_frame_view": (C.c_int, [_H, C.c_int64, C.POINTER(CmFrameView)]),
    "cm_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "cm_host_free": (C.c_int, [C.c_void_p]),
    "cm_run_batch": (C.c_int, [_H, C.POINTER(CmSegment), C.c_int, C.c_void_p]),
    "cm_dev_transform_crop": (C.c_int, [_H, C.POINTER(CmSegment), C.c_int, C.c_void_p]),
    "cm_dev_voxelgrid": (C.c_int, [_H, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "cm_set_zones": (C.c_int, [_H, C.c_int, C.POINTER(CmZone)]),
    "cm_dev_zone_split": (C.c_int, [_H, C.c_void_p, C.c_int64, C.c_void_p]),
    "cm_get_zone_out": (C.c_int, [_H, C.POINTER(CmZoneOut)]),
    "cm_zone_split": (C.c_int, [_H, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "cm_dev_radius_outlier": (C.c_int, [_H, C.c_void_p, C.c_int64, C.c_double, C.c_int, C.c_int, C.c_void_p]),
    "cm_radius_outlier": (C.c_int, [_H, C.c_void_p, C.c_int64, C.c_double, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_int64, C.POINTER(C.c_int64)]),
    "cm_dev_radius_outlier_multi": (C.c_int, [_H, C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.c_double, C.c_int, C.c_int,
                                              C.c_void_p]),
    "cm_radius_outlier_multi": (C.c_int, [_H, C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.c_double, C.c_int, C.c_int,
                                          C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "cm_dev_statistical_outlier": (C.c_int, [_H, C.c_void_p, C.c_int64, C.POINTER(CmSorCfg), C.c_void_p]),
    "cm_dev_statistical_outlier_multi": (C.c_int, [_H, C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.POINTER(CmSorCfg),
                                                   C.c_void_p]),
    "cm_statistical_outlier": (C.c_int, [_H, C.c_void_p, C.c_int64, C.POINTER(CmSorCfg), C.c_void_p, C.c_void_p, C.c_int64,
                                         C.POINTER(C.c_int64)]),
    "cm_statistical_outlier_multi": (C.c_int, [_H, C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.POINTER(CmSorCfg),
                                               C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "cm_get_statistical_out": (C.c_int, [_H, C.POINTER(CmSorOut)]),
    "cm_dev_plane_ransac": (C.c_int, [_H, C.c_void_p, C.c_int64, C.POINTER(CmPlaneCfg), C.POINTER(CmPlane), C.c_void_p]),
    "cm_dev_plane_ransac_multi": (C.c_int, [_H, C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.POINTER(CmPlaneCfg),
                                            C.POINTER(CmPlane), C.c_void_p]),
    "cm_plane_ransac_multi": (C.c_int, [_H, C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.POINTER(CmPlaneCfg), C.POINTER(CmPlane),
                                        C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "cm_plane_ransac": (C.c_int, [_H, C.c_void_p, C.c_int64, C.POINTER(CmPlaneCfg), C.POINTER(CmPlane), C.c_void_p,
                                  C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "cm_dev_proceed_zones": (C.c_int, [_H, C.c_void_p, C.c_int64, C.POINTER(CmProceedCfg), C.POINTER(CmProceedOut), C.c_void_p]),
    "cm_proceed_zones": (C.c_int, [_H, C.c_void_p, C.c_int64, C.POINTER(CmProceedCfg), C.c_void_p, C.c_int64, C.POINTER(C.c_int64),
                                   C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(CmPlane)]),
    "cm_dev_bounds": (C.c_int, [_H, C.c_void_p, C.c_int64, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int64),
                                C.c_void_p]),
    "cm_dev_key_histogram": (C.c_int, [_H, C.c_void_p, C.c_int64, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int,
                                       C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]),
    "cm_dev_route_by_key": (C.c_int, [_H, C.c_void_p, C.c_int64, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                      C.POINTER(C.c_uint64), C.c_int, C.c_int, C.c_void_p]),
    "cm_giant_unique_id": (C.c_int, [C.c_void_p]),
    "cm_giant_create": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "cm_giant_destroy": (C.c_int, [C.c_void_p]),
    "cm_giant_voxelgrid": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(CmGiantInfo), C.c_void_p]),
    "cm_giant_last_error": (C.c_char_p, [C.c_void_p]),
    "cm_sync": (C.c_int, [_H]),
    "cm_get_stats": (C.c_int, [_H, C.POINTER(CmStats)]),
    "cm_get_device_out": (C.c_int, [_H, C.POINTER(CmDeviceOut)]),
    "cm_get_frame_info": (C.c_int, [_H, C.POINTER(CmFrameInfo), C.c_int, C.POINTER(C.c_int)]),
    "cm_launch_count": (C.c_int64, [_H]),
    "cm_set_profiling": (C.c_int, [_H, C.c_int]),
    "cm_stage_ms": (C.c_int, [_H, C.c_char_p, C.POINTER(C.c_float)]),
    "cm_debug_trace": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "cm_stream_create": (C.c_int, [_H, C.POINTER(C.c_void_p)]),
    "cm_stream_destroy": (C.c_int, [_H, C.c_void_p]),
    "cm_stream_sync": (C.c_int, [_H, C.c_void_p]),
    "cm_dev_alloc": (C.c_int, [_H, C.POINTER(C.c_void_p), C.c_size_t]),
    "cm_dev_free": (C.c_int, [_H, C.c_void_p]),
    "cm_memcpy_h2d": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "cm_memcpy_d2h": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "cm_memcpy_d2d": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
}

_LIB = None


def load() -> C.CDLL:
    """Loads the CUDA library. Raises if it has not been built -- there is no fallback implementation."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = os.environ.get("CM_LIB_PATH") or LIB_PATH  # CM_LIB_PATH: a differently tuned build of the same library (experiments)
    if not os.path.exists(path):
        raise RuntimeError(
            "cloud_merger_b200: %s is missing. Build it with `python -m cloud_merger_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback." % path)
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib
