"""cloud_merger_b200 -- B200-native (sm_100a) implementation of cloud_merger's per-frame merge hot path:
per-sensor extrinsic transform -> concat -> PassThrough crop -> VoxelGrid, behind the C ABI of
include/cloud_merger_gpu.h. There is no CPU fallback: loading fails loudly when the CUDA library is missing."""
from .api import (CloudMerger, GiantCloud, giant_unique_id, CloudMergerError, DeviceBuffer, FrameInfo, FrameResult, LAYOUT_LIVOX18, LAYOUT_PACKED16,
                  LAYOUT_PCL32, LAYOUT_VELODYNE22, ROI_PASSES, host_alloc, make_crop_box, make_layout)

__all__ = ["CloudMerger", "GiantCloud", "giant_unique_id", "CloudMergerError", "DeviceBuffer", "FrameInfo", "FrameResult", "LAYOUT_LIVOX18",
           "LAYOUT_PACKED16", "LAYOUT_PCL32", "LAYOUT_VELODYNE22", "ROI_PASSES", "host_alloc", "make_crop_box",
           "make_layout"]
