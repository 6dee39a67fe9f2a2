/*
 * cloud_merger_gpu.h -- C ABI of the B200-native merge hot path of cloud_merger
 * (per-sensor extrinsic transform -> concat -> PassThrough crop -> VoxelGrid).
 *
 * This is the drop-in boundary: plain pointers and sizes, no PCL / Eigen / ROS / torch types. Each entry point names
 * the reference interface it replaces (paths relative to the reference repository timspilak/cloud_merger). The
 * reference-side binding a maintainer adds is shown in INTEGRATION.md and implemented, header-only, in
 * include/cloud_merger_shim.hpp (exact reference signatures: getROI, getCloudPart, fusePointclouds, voxelgrid,
 * transformPointCloud).
 *
 * There is no CPU fallback: every compute entry point needs a CUDA device of compute capability 10.0 (B200) and
 * returns CM_E_CUDA / CM_E_NO_DEVICE otherwise.
 *
 * Threading: cm_submit_cloud is safe to call concurrently for DISTINCT sensor ids of one handle (the reference runs
 * its six sensor callbacks on ros::AsyncSpinner(6), pc_preprocessing_main.cpp:513); cm_merge_frame* may be called
 * from another thread. One handle per GPU.
 */
#ifndef CLOUD_MERGER_GPU_H_
#define CLOUD_MERGER_GPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define CM_API
#else
#define CM_API __attribute__((visibility("default")))
#endif

typedef struct cm_handle_s* cm_handle_t;

/* ---- status codes (the reference functions are void and PCL only warns; every call here returns a code) ---- */
enum {
  CM_OK = 0,
  CM_E_INVALID = 1,     /* bad argument */
  CM_E_CAPACITY = 2,    /* a caller buffer or the handle's configured capacity is too small */
  CM_E_CUDA = 3,        /* CUDA runtime error; cm_last_error(h) has the text */
  CM_E_NO_DEVICE = 4,   /* no CUDA device / not sm_100 */
  CM_E_KEY_RANGE = 5,   /* voxel grid too large for the 64-bit key (more than 2^21 cells on an axis per frame) */
  CM_E_INTERNAL = 6,    /* device-side watchdog tripped (look-back did not make progress) */
  CM_E_NOT_READY = 7    /* no cloud submitted for a sensor named in the mask */
};

/* ---- limits ---- */
#define CM_MAX_PASSES 8
#define CM_MAX_SENSORS 64
#define CM_NO_FIELD (-1)

/* ---- crop: one pcl::PassThrough stage ----
 * Replaces: pcl::PassThrough<pcl::PointXYZI> as configured in getROI (pc_preprocessing_main.cpp:20-40), getCloudPart
 * (:49-59), the z windows of removeGround (:80-92), filter_ROI_R (CloudFusionNode.h:145-190), remove_ground
 * (CloudFusionNode.h:201-216). Limits are float (PCL 1.8.1 setFilterLimits(const float&, const float&)); the window is
 * inclusive; points with a non-finite x, y, z or field value are always removed; negative keeps the outside. Chained
 * passes AND together. With zero passes nothing is removed (the plain cloud_fusion concat, CloudFusionNode.h:59-72). */
typedef struct {
  int32_t axis; /* 0 = "x", 1 = "y", 2 = "z", 3 = "intensity" */
  float lo;
  float hi;
  int32_t negative;
} cm_pass_t;

/* ---- crop: pcl::CropBox stages after the PassThrough chain ----
 * Replaces pcl::CropBox<pcl::PointXYZI> with setMin / setMax / setTranslation / setRotation / setTransform / setNegative
 * (PCL 1.8.1 filters/impl/crop_box.hpp): most often a negative box that removes the vehicle's own body (or a mirror, a roof
 * rack) from the merged cloud, which an AND-ed PassThrough chain cannot express. The boxes run in the given order after the
 * PassThrough chain, each on the previous stage's output, and test the extrinsic-transformed coordinates; survivors keep
 * those coordinates and their input order. Per point and box, as PCL does it: a non-finite x, y or z is removed when the
 * stage's input is not dense (only the first box of a chain without passes sees a non-dense input: the segment's
 * is_dense); then local = transform * p (skipped when transform is the identity within Eigen's 1e-5), local -= translation
 * (when it is not exactly zero), local = inverse(rotation) * local (rotation = roll, pitch, yaw about x, y, z; skipped when
 * it is exactly zero or its inverse is the identity within 1e-5). The point is outside when any local coordinate is below
 * min or above max; negative keeps the outside, otherwise the inside is kept (a NaN coordinate counts as inside). Applies
 * to cm_merge_frame[_async], cm_run_batch and cm_dev_transform_crop; not to zone slicing or the giant-cloud mode.
 * cm_set_crop_boxes with 0 boxes switches them off (the default); NaN limits are refused (CM_E_INVALID). */
#define CM_MAX_CROP_BOXES 8
typedef struct {
  float min[3], max[3];   /* setMin / setMax (PCL's 4th component is not tested) */
  float translation[3];   /* setTranslation */
  float rotation[3];      /* setRotation: roll, pitch, yaw (rad) */
  float transform[12];    /* setTransform: row-major 3x4 of the Eigen::Affine3f; identity = PCL's default */
  int32_t negative;       /* setNegative */
  int32_t reserved;
} cm_crop_box_t;

/* ---- zone slicing: several PassThrough chains over ONE cloud, one ordered output per chain ----
 * Replaces the getCloudPart x5 + z-window sequences the reference runs per sensor cloud in proceedFront / proceedRear /
 * proceedTop / proceedLivox (pc_preprocessing_main.cpp:49-59, 80-92, 228-312: one PassThrough on "x" for
 * [deviation, deviation + length], then "z" for [z_min_g, z_max_g] and for [z_max_g + 0.01, roi_z_max]), filter_ROI_R's
 * three x ranges (CloudFusionNode.h:145-190) and remove_ground's two z windows (:201-216). A zone is a chain of up to
 * CM_MAX_ZONE_PASSES stages; zones may overlap (a point on a shared window end lands in both, as in the reference) and
 * need not cover the cloud; inside a zone the points keep their input order; a zone without stages keeps every point. */
#define CM_MAX_ZONES 16
#define CM_MAX_ZONE_PASSES 4
typedef struct {
  int32_t n_pass;
  cm_pass_t pass[CM_MAX_ZONE_PASSES];
} cm_zone_t;

/* device-resident result of the last zone split on a handle (valid until the next one) */
typedef struct {
  const float* xyzi;                  /* [begin[n_zones]][4] zone 0's points, then zone 1's, ... */
  const uint32_t* src;                /* index of each output point in the input cloud */
  int64_t begin[CM_MAX_ZONES + 1];    /* zone z = [begin[z], begin[z+1]) */
  int32_t n_zones;
  int32_t reserved;
} cm_zone_out_t;

/* RANSAC ground plane: the pcl::SACSegmentation settings of removeGround() (pc_preprocessing_main.cpp:95-108) */
#define CM_SUM4_SSE2 0   /* Eigen packet reductions as an SSE2 build does them: (l0+l2)+(l1+l3) */
#define CM_SUM4_SSE3 1   /* SSE3 and later (haddps): (l0+l1)+(l2+l3) */
#define CM_SUM4_SCALAR 2 /* no vectorisation: ((l0+l1)+l2)+l3 */
typedef struct {
  double distance_threshold; /* seg.setDistanceThreshold (Parameter.h:40: 0.3f) */
  double probability;        /* seg.setProbability (Parameter.h:41: 0.99f) */
  int32_t max_iterations;    /* seg.setMaxIterations (Parameter.h:38: 1000) */
  int32_t optimize;          /* seg.setOptimizeCoefficients (true in the reference) */
  uint32_t seed;             /* 12345 = PCL's sampler (SampleConsensusModel with random == false) */
  int32_t sum_order;         /* CM_SUM4_* */
} cm_plane_cfg_t;
typedef struct {
  int32_t found;        /* 0: segment() failed (fewer than 3 points / no good sample): no inliers */
  int32_t iterations;   /* RandomSampleConsensus iterations_ at exit */
  int32_t draws;        /* three-index draws taken from the sampler (>= iterations: bad samples are redrawn) */
  int32_t best_count;   /* inliers of the RANSAC model */
  int32_t sample[3];    /* the three point indices it was fitted through */
  int32_t reserved;
  float coeff_ransac[4]; /* sac_->getModelCoefficients */
  float coeff[4];        /* what segment() returns: the least-squares refit when optimize != 0 */
  int64_t n_inliers;     /* inliers->indices.size() */
} cm_plane_t;

/* ---- layout of one incoming sensor cloud ----
 * Replaces: the sensor_msgs/PointCloud2 -> pcl::PointCloud<pcl::PointXYZI> deserialisation done by the pcl_ros
 * subscriber (pc_preprocessing_main.cpp:520-525, CloudFusionNode.h:51-56): data[], point_step and the byte offsets of the
 * FLOAT32 fields "x", "y", "z", "intensity". pcl::PointXYZI itself is {32, 0, 4, 8, 16}; packed xyzi is {16, 0, 4, 8, 12}. */
typedef struct {
  int32_t point_step;
  int32_t off_x, off_y, off_z;
  int32_t off_intensity; /* CM_NO_FIELD: no intensity, read as 0 */
  int32_t is_dense;      /* PointCloud2.is_dense: 0 = non-finite points may be present and are left untransformed */
} cm_layout_t;

/* ---- sensor_msgs/PointCloud2 wire adapters (host-only helpers: no device is touched) ----
 * cm_layout_from_pointcloud2 replaces the field lookup of the pcl_ros subscriber (pc_preprocessing_main.cpp:520-525,
 * CloudFusionNode.h:51-56; pcl::createMapping / pcl::fromROSMsg match a field by NAME, DATATYPE and COUNT): given the
 * message's fields[] {name, offset, datatype, count}, point_step, is_bigendian and is_dense it fills the cm_layout_t that
 * cm_submit_cloud needs, so the message's data[] can be handed over as it arrived. "x", "y", "z" must be FLOAT32 (count 1)
 * -> CM_E_INVALID otherwise; an "intensity" field that is missing or not FLOAT32 is treated the way PCL treats an unmatched
 * field (not read; the value is 0) -> off_intensity = CM_NO_FIELD. Big-endian messages are refused (CM_E_INVALID).
 * cm_pointcloud2_describe is the other direction, what pcl::toROSMsg(pcl::PointCloud<pcl::PointXYZI>) would put in the
 * header of the published message (pc_preprocessing_main.cpp:199-220) for n_points records of out_point_step bytes as the
 * kernels write them: height 1, width n, point_step, row_step, little-endian, dense, fields x y z intensity FLOAT32. */
#define CM_PC2_INT8 1
#define CM_PC2_UINT8 2
#define CM_PC2_INT16 3
#define CM_PC2_UINT16 4
#define CM_PC2_INT32 5
#define CM_PC2_UINT32 6
#define CM_PC2_FLOAT32 7
#define CM_PC2_FLOAT64 8
typedef struct {
  const char* name;   /* sensor_msgs/PointField.name */
  uint32_t offset;
  uint8_t datatype;   /* CM_PC2_* == sensor_msgs/PointField constants */
  uint32_t count;
} cm_pc2_field_t;
typedef struct {
  uint32_t height, width, point_step, row_step;
  int32_t is_bigendian, is_dense;
  int32_t n_fields;
  cm_pc2_field_t fields[4];  /* names point to static strings */
} cm_pc2_desc_t;
CM_API int cm_layout_from_pointcloud2(const cm_pc2_field_t* fields, int n_fields, uint32_t point_step, int is_bigendian,
                                      int is_dense, cm_layout_t* out);
CM_API int cm_pointcloud2_describe(int out_point_step, int64_t n_points, cm_pc2_desc_t* out);

/* ---- one segment of a device-resident batch: one sensor cloud of one frame ---- */
typedef struct {
  const void* data;   /* DEVICE pointer, 16-byte aligned */
  int64_t n_points;
  cm_layout_t layout;
  int32_t sensor;     /* which extrinsic (cm_set_extrinsic) applies */
  int32_t frame;      /* 0-based frame number inside the batch; segments must be ordered by frame, then concat order */
} cm_segment_t;

/* ---- creation-time configuration ---- */
typedef struct {
  int32_t device;                 /* CUDA device ordinal */
  int32_t max_sensors;            /* sensors per frame (<= CM_MAX_SENSORS) */
  int64_t max_points_per_sensor;  /* capacity of one submitted cloud (host path) */
  int32_t max_point_step;         /* largest point_step the host path will see (bytes) */
  int32_t frames_in_flight;       /* host-path pipeline depth: 1..8 */
  int64_t max_batch_points;       /* capacity (points) of one device-resident batch; 0 = max_sensors*max_points_per_sensor */
  int32_t max_batch_frames;       /* frames per device-resident batch (>= 1) */
  int32_t max_batch_segments;     /* segments per batch; 0 = max_batch_frames*max_sensors */
  int32_t out_point_step;         /* 16 = packed float4 xyzi; 32 = pcl::PointXYZI record (pad@12 = 1.0f) so pcl::toROSMsg is a memcpy */
  int32_t reserved;
} cm_config_t;

/* ---- per-run statistics (metrics the reference only prints via ROS_INFO) ---- */
typedef struct {
  int64_t points_in;       /* points submitted */
  int64_t survivors;       /* points after the crop */
  int64_t voxels_out;      /* voxels emitted */
  int32_t frames;          /* frames in the run */
  int32_t key_bits;        /* significant voxel-key bits that were sorted */
  int32_t sort_passes;     /* radix passes executed */
  int32_t key_bytes;       /* 4 or 8 */
  int32_t pcl_overflow;    /* number of frames for which PCL 1.8.1 would refuse ("Leaf size is too small") */
  int32_t device_error;    /* 0 or a CM_E_* raised on the device */
  float gpu_ms;            /* device time of the run between its first and last kernel (CUDA events) */
  float reserved;
} cm_stats_t;

/* ---- per-frame results of a batch (device arrays are indexed by these) ---- */
typedef struct {
  int64_t survivor_begin, survivor_end; /* this frame's slice of the merged, cropped cloud */
  int64_t voxel_begin, voxel_end;       /* this frame's slice of the voxel output */
  int32_t min_b[3], max_b[3], div_b[3]; /* pcl::VoxelGrid getMinBoxCoordinates / getMaxBoxCoordinates / getNrDivisions */
  int32_t pcl_overflow;                 /* 1: PCL 1.8.1 would have returned the input unchanged for this frame */
} cm_frame_info_t;

/* ---- device-resident outputs of the last batch run on a handle (valid until the next run) ---- */
typedef struct {
  const float* survivor_xyzi;    /* [survivors][4] merged + cropped cloud, transform applied (concat order); dense copy made by this call */
  const uint32_t* survivor_src;  /* [survivors] index of each survivor in its frame's un-cropped concatenation */
  const uint32_t* survivor_slot; /* [survivors] slot of each survivor (NULL when the cloud never went through the crop: slot == index) */
  const float* slot_xyzi;        /* the kernels' own layout: survivors compacted tile by tile, addressed by slot */
  const void* sorted_key;        /* [survivors] voxel keys ascending (uint32 or uint64, see key_bytes) */
  const uint32_t* sorted_point;  /* [survivors] SLOT of the point belonging to sorted_key[i] (voxel membership) */
  const void* voxel_xyzi;        /* [voxels] centroids, out_point_step bytes each */
  const uint32_t* voxel_count;   /* [voxels] points per voxel */
  const uint64_t* voxel_idx;     /* [voxels] PCL's voxel index idx = i + j*div_x + k*div_x*div_y (64-bit) */
  int32_t key_bytes;
  int32_t key_idx_bits;          /* key = (frame << key_idx_bits) | idx */
} cm_device_out_t;

/* ---- host-side result of one merged frame ---- */
typedef struct {
  /* caller buffers (any may be NULL to skip that output) and their capacities in elements */
  void* voxel_xyzi;        int64_t voxel_capacity;     /* out_point_step bytes per voxel */
  uint32_t* voxel_count;
  uint64_t* voxel_idx;
  float* survivor_xyzi;    int64_t survivor_capacity;  /* [survivors][4] the merged cropped cloud (== /points_no_ground input of voxelgrid) */
  uint32_t* survivor_src;
  /* filled by the call */
  int64_t n_voxels;
  int64_t n_survivors;
  cm_frame_info_t info;
} cm_frame_out_t;

/* ---- lifecycle ---- */
CM_API int cm_create(const cm_config_t* cfg, cm_handle_t* out);
CM_API int cm_destroy(cm_handle_t h);
CM_API const char* cm_strerror(int code);
CM_API const char* cm_last_error(cm_handle_t h);
CM_API const char* cm_version(void);
CM_API int cm_device_count(void);

/* ---- configuration ----
 * cm_set_extrinsic replaces the tf::Transform -> Eigen::Affine3f argument of pcl_ros::transformPointCloud
 * (pc_preprocessing_main.cpp:320-322 and the five other callbacks; CloudFusionNode.h:506-534). m is a 4x4 float matrix;
 * col_major != 0 reads Eigen::Matrix4f::data() order. Only rows 0..2 are used (rigid / affine transform).
 * cm_set_extrinsic_tf builds it the way pcl_ros does from a tf::Transform: double quaternion (x, y, z, w) + origin,
 * narrowed to float, Eigen 3.3 toRotationMatrix. */
CM_API int cm_set_extrinsic(cm_handle_t h, int sensor, const float* m16, int col_major);
CM_API int cm_set_extrinsic_tf(cm_handle_t h, int sensor, const double* quat_xyzw, const double* origin_xyz);
CM_API int cm_get_extrinsic(cm_handle_t h, int sensor, float* m12_row_major);
/* cm_set_crop replaces the PassThrough chains (see cm_pass_t). Defaults = getROI with Parameter.h:31-35. */
CM_API int cm_set_crop(cm_handle_t h, int n_pass, const cm_pass_t* passes);
/* cm_set_crop_boxes replaces the pcl::CropBox stages that follow the PassThrough chain (see cm_crop_box_t). */
CM_API int cm_set_crop_boxes(cm_handle_t h, int n_boxes, const cm_crop_box_t* boxes);
/* cm_set_voxel replaces voxel_grid.setLeafSize / setDownsampleAllData / setMinimumPointsNumberPerVoxel
 * (pc_preprocessing_main.cpp:171-175). Defaults: leaf 0.1, min_points 2, downsample_all 1 (Parameter.h:27-28). */
CM_API int cm_set_voxel(cm_handle_t h, const float* leaf3, int min_points, int downsample_all);
/* Single-giant-cloud mode (one cloud partitioned by voxel-key range over several GPUs): the bounding box pcl::getMinMax3D
 * would find on the WHOLE cloud, all-reduced by the caller. The next cm_dev_voxelgrid calls fold it into the local box, so
 * every rank builds the same grid (same min_b / div_b / voxel indices). NULL, NULL switches it off. */
CM_API int cm_set_voxel_bounds(cm_handle_t h, const float* min3, const float* max3);
/* PCL 1.8.1 returns the input cloud unchanged when dx*dy*dz > INT32_MAX. mode 0 (default): keep going with the 64-bit
 * key and report it in cm_frame_info_t.pcl_overflow; mode 1: behave like PCL (the frame's output is its cropped cloud).
 * A frame whose grid is beyond the key range (more than 2^21 cells on an axis, or a cell origin beyond +-2^30) fails with
 * CM_E_KEY_RANGE, except in mode 1 when PCL refuses it too: cm_wait_frame / cm_merge_frame then return its cropped cloud
 * (in a device batch its voxels are meaningless and frame_info.pcl_overflow says so). */
CM_API int cm_set_overflow_mode(cm_handle_t h, int mode);

/* ---- host path: one frame at a time, callable from the ROS callbacks ----
 * cm_submit_cloud replaces the body of callbackFrontRight .. callbackFrontMiddle up to the hand-off into the globals
 * (pc_preprocessing_main.cpp:318-337 ...) and add_*_velodyne (CloudFusionNode.h:506-534): it takes the raw point records,
 * copies them to the device asynchronously and returns. stamp feeds operator+='s "newest stamp" rule.
 * Which cloud of a sensor a frame is merged from, when the sensor delivers more than one between two merges
 * (cm_set_submit_policy):
 *   CM_SUBMIT_LATEST_WINS (default)  the newest one -- what my_cloud_fusion does (add_*_velodyne overwrites its member cloud on
 *                                    every callback, CloudFusionNode.h:506-534);
 *   CM_SUBMIT_FIRST_WINS             the first one after the previous merge -- pcl_preprocessing's flag gate
 *                                    `if (!flag_x) { store; flag_x = true; }` (pc_preprocessing_main.cpp:330-336): later clouds
 *                                    are dropped (the call returns CM_OK without copying) until the frame has been merged.
 * Every submission ends with the next merge: clouds of sensors in the merge mask are consumed, clouds of other sensors are
 * discarded. */
#define CM_SUBMIT_LATEST_WINS 0
#define CM_SUBMIT_FIRST_WINS 1
CM_API int cm_set_submit_policy(cm_handle_t h, int policy);
CM_API int cm_submit_cloud(cm_handle_t h, int sensor, const void* data, int64_t n_points, const cm_layout_t* layout,
                           uint64_t stamp);
/* Same, for a caller buffer that is page-locked (cm_host_alloc / cudaHostRegister) and stays untouched until the frame it
 * belongs to has been waited for: the copy goes straight from the caller's memory, with no staging memcpy. */
CM_API int cm_submit_cloud_pinned(cm_handle_t h, int sensor, const void* data, int64_t n_points,
                                  const cm_layout_t* layout, uint64_t stamp);
/* Several page-locked clouds of one frame at once (a rosbag replay, or a driver that delivers all sensors together):
 * the same as `count` calls of cm_submit_cloud_pinned, except that clouds which follow each other in host memory and
 * belong to consecutive sensor ids are copied with one transfer (into a per-frame arena of the handle, so the run shares
 * no device bytes with single submissions of its members). stamps may be NULL. */
CM_API int cm_submit_clouds_pinned(cm_handle_t h, int count, const int* sensors, const void* const* data,
                                   const int64_t* n_points, const cm_layout_t* layouts, const uint64_t* stamps);
/* cm_merge_frame replaces fusePointclouds + voxelgrid (pc_preprocessing_main.cpp:131-177, main loop :574-578):
 * merges the latest cloud of every sensor in sensor_mask (bit s = sensor s, concat order = ascending sensor id),
 * crops, voxel-filters and copies the results into the caller's buffers. Blocks until the results are on the host.
 * Sensors in the mask that have nothing submitted are skipped (the reference's optional top sensor, :134-136);
 * *out_used_mask (may be NULL) receives the sensors actually merged. The merged clouds are consumed (flags reset). */
CM_API int cm_merge_frame(cm_handle_t h, uint64_t sensor_mask, cm_frame_out_t* out, uint64_t* out_used_mask,
                          uint64_t* out_stamp);
/* Pipelined form: cm_merge_frame_async enqueues the work and returns a ticket; cm_wait_frame blocks on that ticket and
 * copies out. Up to frames_in_flight tickets may be outstanding. The voxel outputs travel to page-locked host memory on the
 * frame's own stream (sized on the device), so cm_wait_frame is ONE synchronisation followed by host memcpys; only the
 * optional survivor outputs cost a second device round trip. */
CM_API int cm_merge_frame_async(cm_handle_t h, uint64_t sensor_mask, int64_t* ticket);
CM_API int cm_wait_frame(cm_handle_t h, int64_t ticket, cm_frame_out_t* out, uint64_t* out_used_mask,
                         uint64_t* out_stamp);
/* Zero-copy form of cm_wait_frame: instead of copying the voxels into caller buffers it hands out pointers into the
 * library's own page-locked result mirrors of that frame -- the frame's stream wrote them there itself. The view stays valid
 * until frames_in_flight further frames have been merged on the handle (the frame slot is reused then). With PCL-like
 * overflow mode and a frame PCL would refuse, use cm_wait_frame (the result is the merged cloud, which has no mirror). */
typedef struct {
  const void* voxel_xyzi;       /* HOST, page-locked: [n_voxels] records of out_point_step bytes */
  const uint32_t* voxel_count;  /* HOST [n_voxels] */
  const uint64_t* voxel_idx;    /* HOST [n_voxels] */
  int64_t n_voxels, n_survivors;
  cm_frame_info_t info;
  uint64_t used_mask, stamp;
} cm_frame_view_t;
CM_API int cm_wait_frame_view(cm_handle_t h, int64_t ticket, cm_frame_view_t* view);
/* Pinned host memory for callers that want true asynchronous H2D/D2H (e.g. the ROS message buffers). The pages are placed
 * on the NUMA node of the CURRENT CUDA device (cudaSetDevice before the call; the library's own staging buffers follow the
 * handle's device) where the platform tells which node that is -- eight processes feeding eight GPUs from arenas that all
 * landed on one node share one set of memory controllers. CM_NO_NUMA=1 in the environment switches the placement off. */
CM_API int cm_host_alloc(void** p, size_t bytes);
CM_API int cm_host_free(void* p);

/* ---- device path: a batch of frames whose raw clouds already sit in device memory ----
 * One call runs the whole path for every frame of the batch (F frames x S sensors = n_segments segments) with a fixed
 * number of kernel launches; stream is a cudaStream_t (NULL = legacy default stream). Results stay on the device
 * (cm_get_device_out) with per-frame slices in cm_get_frame_info. */
CM_API int cm_run_batch(cm_handle_t h, const cm_segment_t* segments, int n_segments, void* stream);
/* Stage-level entry points on device pointers (benchmarks, tests, and the building blocks of the shim):
 *  cm_dev_transform_crop: the fused unpack + transform + crop + stable compaction only
 *      (== transformPointCloud + getROI + operator+=); results in cm_get_device_out().survivor_*.
 *  cm_dev_voxelgrid: VoxelGrid only on n packed float4 xyzi points already on the device (== voxelgrid()). */
CM_API int cm_dev_transform_crop(cm_handle_t h, const cm_segment_t* segments, int n_segments, void* stream);
CM_API int cm_dev_voxelgrid(cm_handle_t h, const float* xyzi_dev, int64_t n_points, int is_dense, void* stream);
/* Zone slicing (see cm_zone_t). cm_set_zones configures the chains; cm_dev_zone_split runs them over n packed float4
 * xyzi points on the device -- or, with xyzi_dev == NULL, over the merged cropped cloud of the handle's last
 * cm_dev_transform_crop / cm_run_batch (== getROI's output, the input of getCloudPart in the reference);
 * cm_get_zone_out waits and returns the device arrays. cm_zone_split is the host-buffer form (H2D, split, D2H):
 * out_begin receives n_zones + 1 offsets; returns CM_E_CAPACITY (and the needed size in out_begin[n_zones]) when the
 * zones together do not fit `capacity` points. */
CM_API int cm_set_zones(cm_handle_t h, int n_zones, const cm_zone_t* zones);
CM_API int cm_dev_zone_split(cm_handle_t h, const float* xyzi_dev, int64_t n_points, void* stream);
CM_API int cm_get_zone_out(cm_handle_t h, cm_zone_out_t* out);
CM_API int cm_zone_split(cm_handle_t h, const float* xyzi_host, int64_t n_points, float* out_xyzi, uint32_t* out_src,
                         int64_t capacity, int64_t* out_begin);
/* Radius outlier removal. Replaces outlierRemoval() (pc_preprocessing_main.cpp:184-192, called from removeGround :119):
 * pcl::RadiusOutlierRemoval<pcl::PointXYZI> with setRadiusSearch(radius), setMinNeighborsInRadius(min_neighbors),
 * keep_organized false (Parameter.h:23-24: 0.15 m, 1). PCL 1.8.1 keeps a point iff MORE than min_neighbors points -- the
 * point itself included -- lie strictly inside the radius (float squared distances, FLANN's order); negative != 0 keeps
 * the others. Non-finite points are never kept. Survivors keep their input order.
 *  cm_dev_radius_outlier: n packed float4 xyzi points on the device; results through cm_get_zone_out (one zone: xyzi +
 *      the index of every survivor in the input). Uses the handle's batch workspace (the previous run's device outputs
 *      are overwritten). CM_E_KEY_RANGE when the radius is too small for the extent of the cloud: the call itself returns
 *      it when the cell grid exceeds the key range (more than 2^21 cells on an axis, a coordinate beyond 2^30 cells);
 *      cm_get_zone_out returns it when a point lies 2^14 cells or more from the origin (the cell margin only covers
 *      less, so the neighbour counts are not guaranteed). The next call on the handle is not affected.
 *  cm_radius_outlier: host buffers in and out; *n_out receives the number of survivors (also on CM_E_CAPACITY). */
CM_API int cm_dev_radius_outlier(cm_handle_t h, const float* xyzi_dev, int64_t n_points, double radius,
                                 int min_neighbors, int negative, void* stream);
CM_API int cm_radius_outlier(cm_handle_t h, const float* xyzi_host, int64_t n_points, double radius, int min_neighbors,
                             int negative, float* out_xyzi, uint32_t* out_idx, int64_t capacity, int64_t* n_out);
/* Several independent clouds in one pass (the per-zone outlierRemoval calls of one proceedX): cloud k = the points
 * [begin[k], begin[k+1]) of the array (begin[0] == 0, n_clouds <= CM_MAX_ZONES and <= the handle's max_batch_frames).
 * Every cloud has its own cell grid and neighbours are never counted across clouds. Results: zone k of cm_get_zone_out =
 * the survivors of cloud k (src = index in the whole array); the host form writes n_clouds + 1 offsets to out_begin.
 * CM_E_KEY_RANGE as for one cloud, when any of the clouds is too large for the radius. */
CM_API int cm_dev_radius_outlier_multi(cm_handle_t h, const float* xyzi_dev, const int64_t* begin, int n_clouds,
                                       double radius, int min_neighbors, int negative, void* stream);
CM_API int cm_radius_outlier_multi(cm_handle_t h, const float* xyzi_host, const int64_t* begin, int n_clouds, double radius,
                                   int min_neighbors, int negative, float* out_xyzi, uint32_t* out_idx, int64_t capacity,
                                   int64_t* out_begin);
/* Statistical outlier removal: pcl::StatisticalOutlierRemoval<pcl::PointXYZI> with setMeanK(mean_k),
 * setStddevMulThresh(std_mul), setNegative(negative), keep_organized false (PCL 1.8.1 applyFilterIndices). Every finite
 * point gets the mean of the square roots of its mean_k nearest squared distances (exact search, float distances in
 * FLANN's order, double sum in ascending order, stored as a float); a non-finite point gets 0. Over every cloud, in index
 * order and in double: mean and stddev of those values over the finite points, threshold = mean + std_mul * stddev; a
 * point is removed iff its value > threshold (negative != 0: iff <=). Survivors keep their input order.
 * Documented deviations: the input is always treated as non-dense; a cloud with 0 < finite points <= mean_k (PCL reads
 * past its neighbour vectors there) keeps every point, whatever negative is, and is flagged too_few.
 *  cm_dev_statistical_outlier[_multi]: packed float4 xyzi points on the device (clouds as for the radius outlier removal:
 *      cloud k = [begin[k], begin[k+1]), n_clouds <= CM_MAX_ZONES and <= max_batch_frames, no neighbours across clouds).
 *      Survivors through cm_get_zone_out (zone k = those of cloud k, src = index in the whole array), the per-point values
 *      and per-cloud statistics through cm_get_statistical_out. mean_k outside 1 .. CM_SOR_MAX_K, a NaN std_mul or an
 *      unknown sqrt_mode -> CM_E_INVALID. Uses the handle's batch workspace, like the radius outlier removal.
 *  cm_statistical_outlier[_multi]: host buffers in and out (CM_E_CAPACITY with the needed size in *n_out /
 *      out_begin[n_clouds]). */
#define CM_SOR_MAX_K 127
#define CM_SOR_SQRT_FLOAT 0   /* the unqualified sqrt of PCL's loop resolves to std::sqrt(float) */
#define CM_SOR_SQRT_DOUBLE 1  /* ... to ::sqrt(double) on the promoted value */
typedef struct {
  int32_t mean_k;     /* setMeanK, 1 .. CM_SOR_MAX_K */
  int32_t negative;   /* setNegative */
  int32_t sqrt_mode;  /* CM_SOR_SQRT_* */
  int32_t reserved;
  double std_mul;     /* setStddevMulThresh */
} cm_sor_cfg_t;
#define CM_SOR_SUM_SERIAL 1     /* sum_path bit: the sum of the values was formed by the serial chain in index order */
#define CM_SOR_SQ_SUM_SERIAL 2  /* ... the sum of their squares (otherwise: an exact parallel sum, the same bits) */
typedef struct {
  double mean, stddev, threshold; /* PCL's distance statistics of the cloud (NaN threshold: every point is kept) */
  int64_t n_valid;                /* finite points */
  int32_t too_few;                /* 0 < n_valid <= mean_k: no search, every point kept, values 0 */
  int32_t sum_path;               /* CM_SOR_*SERIAL bits */
} cm_sor_stats_t;
typedef struct {
  const float* distances;         /* device [n_points]: the value of every input point, in input order */
  int64_t n_points;
  int32_t n_clouds;
  int32_t reserved;
  float knn_ms, sums_ms;          /* GPU time of the neighbour search and of the sums (cm_set_profiling on; -1 otherwise) */
  cm_sor_stats_t cloud[CM_MAX_ZONES];
} cm_sor_out_t;
CM_API int cm_dev_statistical_outlier(cm_handle_t h, const float* xyzi_dev, int64_t n_points, const cm_sor_cfg_t* cfg,
                                      void* stream);
CM_API int cm_dev_statistical_outlier_multi(cm_handle_t h, const float* xyzi_dev, const int64_t* begin, int n_clouds,
                                            const cm_sor_cfg_t* cfg, void* stream);
CM_API int cm_statistical_outlier(cm_handle_t h, const float* xyzi_host, int64_t n_points, const cm_sor_cfg_t* cfg,
                                  float* out_xyzi, uint32_t* out_idx, int64_t capacity, int64_t* n_out);
CM_API int cm_statistical_outlier_multi(cm_handle_t h, const float* xyzi_host, const int64_t* begin, int n_clouds,
                                        const cm_sor_cfg_t* cfg, float* out_xyzi, uint32_t* out_idx, int64_t capacity,
                                        int64_t* out_begin);
/* waits for the last statistical outlier removal on the handle; the device array stays valid until the next one */
CM_API int cm_get_statistical_out(cm_handle_t h, cm_sor_out_t* out);
/* RANSAC ground plane. Replaces the pcl::SACSegmentation + pcl::ExtractIndices block of removeGround()
 * (pc_preprocessing_main.cpp:95-117): SACMODEL_PLANE, SAC_RANSAC (setAxis / setEpsAngle are ignored by that model, as in
 * PCL). The three-index draws are PCL 1.8.1's -- boost::mt19937 seeded with cfg->seed, uniform_int<>(0, INT_MAX), the
 * partial shuffle of drawIndexSample -- and are scored on the GPU a batch at a time; the host applies PCL's stopping rule
 * to the batch in draw order, so model, iteration count and inliers are those of PCL's sequential loop. With optimize the
 * least-squares refit follows (float running sums in inlier order as computeMeanAndCovarianceMatrix forms them, pcl::eigen33
 * on the host) and the inliers are selected again.
 * Zone slicing, radius outlier removal and the plane search write their results into the handle's zone outputs
 * (cm_get_zone_out): an input cloud that lies there is refused with CM_E_INVALID -- chain stages over separate handles.
 *  cm_dev_plane_ransac: n packed float4 xyzi points on the device; blocks until the model is known. Results: *out, and
 *      through cm_get_zone_out two zones in input order -- zone 0 the inliers (ground_cloud), zone 1 the rest
 *      (no_ground_cloud before outlierRemoval), src = index in the input.
 *  cm_plane_ransac: host buffers; out_begin receives 3 offsets (inliers = [0, out_begin[1]), rest up to out_begin[2]). */
CM_API int cm_dev_plane_ransac(cm_handle_t h, const float* xyzi_dev, int64_t n_points, const cm_plane_cfg_t* cfg,
                               cm_plane_t* out, void* stream);
/* Several independent plane searches in one pass (the ground zones of one sensor cloud: five RANSACs per proceedX,
 * pc_preprocessing_main.cpp:228-312): cloud k = the points [begin[k], begin[k+1]) of xyzi_dev (begin[0] == 0),
 * n_clouds <= CM_MAX_ZONES / 2. Every batch of hypotheses, the selection and the refit cover all clouds at once, so the
 * call costs about as much as one search. out[n_clouds]; cm_get_zone_out then holds 2 * n_clouds zones: zone 2k = the
 * inliers of cloud k, zone 2k + 1 = its other points (src = index in xyzi_dev, i.e. begin[k] + index in the cloud). */
CM_API int cm_dev_plane_ransac_multi(cm_handle_t h, const float* xyzi_dev, const int64_t* begin, int n_clouds,
                                     const cm_plane_cfg_t* cfg, cm_plane_t* out, void* stream);
/* host-buffer form of the above: out_begin receives 2 * n_clouds + 1 offsets into out_xyzi / out_idx */
CM_API int cm_plane_ransac_multi(cm_handle_t h, const float* xyzi_host, const int64_t* begin, int n_clouds,
                                 const cm_plane_cfg_t* cfg, cm_plane_t* out, float* out_xyzi, uint32_t* out_idx,
                                 int64_t capacity, int64_t* out_begin);
CM_API int cm_plane_ransac(cm_handle_t h, const float* xyzi_host, int64_t n_points, const cm_plane_cfg_t* cfg,
                           cm_plane_t* out, float* out_xyzi, uint32_t* out_idx, int64_t capacity, int64_t* out_begin);
/* ---- the body of a proceedX in ONE call ----
 * Replaces what proceedFront / proceedRear / callbackTopMiddle / callbackFrontMiddle do after getROI
 * (pc_preprocessing_main.cpp:228-312, :428-446, :474-497): for every part of the sensor's zone table
 *     getCloudPart(cloud_ROI_ptr, part, length, deviation);                                   x in [deviation, deviation + length]
 *     removeGround(part, no_ground, ground, -z_max_ground, z_max_ground, max_angle);          :71-122
 *         z windows [-z_max_ground, z_max_ground] and [z_max_ground + 0.01, roi_z_max], RANSAC plane + ExtractIndices on the
 *         lower one, outlierRemoval of its non-ground points, the upper window appended
 *     no_ground += ...; ground += ...;
 * and a part with ground_removal == 0 is appended to the no-ground cloud as it is (the near range of the top sensor,
 * :444-446). One zone-slicing pass for every window, one multi-cloud plane search, one multi-cloud outlier removal and the
 * appends, all on one handle and one stream, device-resident in between (the host only sees the stopping rule of the plane
 * search, the 3 x 3 refit and the sizes). Needs max_batch_frames >= the number of ground-removal parts.
 *  cm_dev_proceed_zones  n packed float4 xyzi points on the device (the ROI cloud); results stay on the device (valid until
 *                        the next cm_*proceed_zones on the handle);
 *  cm_proceed_zones      host buffers in and out; *n_no_ground / *n_ground receive the sizes (also on CM_E_CAPACITY). */
#define CM_MAX_PROCEED_PARTS 8
typedef struct {
  float length, deviation;  /* getCloudPart arguments */
  float z_max_ground;       /* ground window |z| <= z_max_ground */
  int32_t ground_removal;   /* 1: removeGround on the part; 0: the part goes to the no-ground cloud unchanged */
} cm_proceed_part_t;
typedef struct {
  int32_t n_parts;
  int32_t min_neighbors;    /* outlierRemoval: Parameter.h:24 */
  cm_proceed_part_t part[CM_MAX_PROCEED_PARTS];
  float roi_z_max;          /* upper end of the no-ground window (Parameter.h:35) */
  float reserved;
  double radius;            /* outlierRemoval: Parameter.h:23 */
  cm_plane_cfg_t plane;     /* SACSegmentation settings (Parameter.h:38-42) */
} cm_proceed_cfg_t;
typedef struct {
  const float* no_ground_xyzi;  /* DEVICE [n_no_ground][4] */
  const float* ground_xyzi;     /* DEVICE [n_ground][4] */
  int64_t n_no_ground, n_ground;
  cm_plane_t plane[CM_MAX_PROCEED_PARTS];  /* the model of every ground-removal part, in part order */
  int32_t n_planes;
  int32_t host_syncs;           /* device round trips the call needed (diagnostic) */
} cm_proceed_out_t;
CM_API int cm_dev_proceed_zones(cm_handle_t h, const float* roi_xyzi_dev, int64_t n_points, const cm_proceed_cfg_t* cfg,
                                cm_proceed_out_t* out, void* stream);
CM_API int cm_proceed_zones(cm_handle_t h, const float* roi_xyzi_host, int64_t n_points, const cm_proceed_cfg_t* cfg,
                            float* out_no_ground, int64_t no_ground_capacity, int64_t* n_no_ground, float* out_ground,
                            int64_t ground_capacity, int64_t* n_ground, cm_plane_t* out_planes);

/* ---- single giant cloud over several GPUs (BASELINE config 4): device-side pieces of the voxel-key range partition ----
 * The reference has no counterpart (one process). Every rank holds a block of the cloud; all ranks must build the SAME
 * voxel grid, a voxel must not straddle ranks, and the rank outputs concatenated in rank order must be PCL's order:
 *  cm_dev_bounds         pcl::getMinMax3D of the local block (blocking; the caller all-reduces min / max);
 *  cm_dev_key_histogram  histogram (uint64 bins on the device, equal key width, *out_bin_width) of the PCL voxel index
 *                        idx = i + j*div_x + k*div_x*div_y on the grid of the GLOBAL box (the caller all-reduces it and
 *                        cuts it into balanced key ranges);
 *  cm_dev_route_by_key   groups the local points by destination: part r owns idx in [splitters[r-1], splitters[r])
 *                        (n_parts - 1 splitters; non-finite points go to invalid_part); source order is kept inside a
 *                        part. Results through cm_get_zone_out (zone r = the send buffer for rank r).
 * The owning rank then runs cm_set_voxel_bounds + cm_dev_voxelgrid on what it received. Leaf = cm_set_voxel. */
CM_API int cm_dev_bounds(cm_handle_t h, const float* xyzi_dev, int64_t n_points, float* min3, float* max3,
                         int64_t* n_finite, void* stream);
CM_API int cm_dev_key_histogram(cm_handle_t h, const float* xyzi_dev, int64_t n_points, const float* min3,
                                const float* max3, int bins, uint64_t* hist_dev, uint64_t* out_bin_width, void* stream);
CM_API int cm_dev_route_by_key(cm_handle_t h, const float* xyzi_dev, int64_t n_points, const float* min3,
                               const float* max3, const uint64_t* splitters, int n_parts, int invalid_part, void* stream);
/* ---- the whole giant-cloud VoxelGrid behind ONE call, C++ + NCCL (BASELINE config 4) ----
 * One process per GPU; every rank holds a block of the cloud in device memory. cm_giant_voxelgrid does, on `stream`:
 *   bounding box of the block -> ncclAllReduce (max of order-preserving encodings) -> PCL's grid on the global box, ON THE DEVICE
 *   -> histogram of the voxel index -> ncclAllReduce (sum) -> balancing splitters, ON THE DEVICE -> group the block by
 *   destination rank (source order kept) -> ncclAllGather of the per-destination counts -> ONE exchange, 16 bytes per
 *   point (see CM_GIANT_EXCHANGE_* below: stores into the owners' buffers over NVLink from inside the grouping kernel, or a
 *   grouped ncclSend / ncclRecv) -> the single-GPU VoxelGrid on what arrived, with the global box folded in so that every
 *   rank builds the same grid.
 * The host is needed twice: for the counts (they size the VoxelGrid launches; NCCL also takes them as host arguments) and
 * for the final report. Calls on one object must be stream-ordered on every rank (the same stream, or streams the caller
 * orders): a peer may store into this rank's receive buffer as soon as this rank has entered the next call.
 * A voxel never straddles ranks, and the rank outputs (cm_get_device_out on each rank: voxel_xyzi / voxel_count / voxel_idx)
 * concatenated in rank order are PCL's order. Leaf and min_points: cm_set_voxel on the handle. The handle's
 * max_batch_points bounds what a rank may RECEIVE (balanced splitters give ~n / world; size it with headroom).
 * NCCL is loaded at run time (libnccl.so.2 -- the copy already in the process if there is one, e.g. PyTorch's);
 * communicator bootstrap: rank 0 calls cm_giant_unique_id and ships the 128 bytes to every rank by any means.
 * With nccl_id == NULL and world > 1 the object is "dry": no communicator, the collectives are identities, and
 * cm_giant_voxelgrid stops after the grouping (results through cm_get_zone_out) -- the routing can be tested on one GPU. */
typedef struct cm_giant_s* cm_giant_t;
#define CM_GIANT_ID_BYTES 128
/* The exchange: PEER = the grouping kernel stores every point straight into its owner's receive buffer over NVLink (the
 * buffers are mapped into every rank through CUDA IPC at cm_giant_create; one kernel is scatter and all-to-all at once,
 * closed by a one-word all-reduce); NCCL = grouped into a local send buffer, then one grouped ncclSend / ncclRecv. PEER is
 * chosen when every rank could map every peer (one process per GPU on an NVLink box); CM_GIANT_NO_P2P=1 in the environment
 * forces NCCL. Both deliver the same points in the same order. */
#define CM_GIANT_EXCHANGE_NONE 0
#define CM_GIANT_EXCHANGE_NCCL 1
#define CM_GIANT_EXCHANGE_PEER 2
typedef struct {
  int64_t points_local, points_received, points_sent_away, points_total_finite;
  int64_t voxels_local;            /* filled by cm_giant_report */
  uint64_t splitter[CM_MAX_ZONES]; /* world - 1 valid entries */
  float min_p[3], max_p[3];        /* global bounding box */
  int32_t min_b[3], div_b[3];      /* PCL's grid on it */
  int32_t key_bits, host_syncs;
  int32_t exchange;                /* CM_GIANT_EXCHANGE_*: how the points reached their owners in this call */
  int32_t reserved;
  float stage_ms[4];               /* with cm_set_profiling(h, 1) (the call then blocks until its last kernel is done): device
                                    * time of [0] bounds + histogram + splitters, [1] grouping (mask, count, scan, offsets),
                                    * [2] the exchange, [3] the local VoxelGrid; else zeros */
  int64_t send_begin[CM_MAX_ZONES + 1]; /* where the points for rank r start in the grouped array */
} cm_giant_info_t;
CM_API int cm_giant_unique_id(void* id_bytes);
CM_API int cm_giant_create(cm_handle_t h, int rank, int world, const void* nccl_id, cm_giant_t* out);
CM_API int cm_giant_destroy(cm_giant_t g);
CM_API int cm_giant_voxelgrid(cm_giant_t g, const float* local_xyzi_dev, int64_t n_local, cm_giant_info_t* info, void* stream);
CM_API const char* cm_giant_last_error(cm_giant_t g);

/* Blocks until the last run on the handle finished, then reports. */
CM_API int cm_sync(cm_handle_t h);
CM_API int cm_get_stats(cm_handle_t h, cm_stats_t* out);
CM_API int cm_get_device_out(cm_handle_t h, cm_device_out_t* out);
CM_API int cm_get_frame_info(cm_handle_t h, cm_frame_info_t* out, int capacity, int* n_frames);
/* Number of kernel launches the last run enqueued (the caller's "gpu_launches" evidence). Only launches that happened are
 * counted. After cm_[dev_]zone_split: the split (3, or 1 without points), plus 1 once cm_get_zone_out has repeated the
 * scatter into grown outputs. After cm_[dev_]plane_ransac[_multi]: the whole call, scoring rounds, refit sums, select and
 * compaction. After cm_[dev_]radius_outlier[_multi] and cm_[dev_]statistical_outlier[_multi]: the filter up to its mask,
 * without the compaction. After cm_dev_route_by_key: the mask kernel and the split. After cm_[dev_]proceed_zones: the
 * radius outlier removal when a part removes ground, else the zone split. After cm_giant_voxelgrid: its local VoxelGrid. */
CM_API int64_t cm_launch_count(cm_handle_t h);
/* Device time (ms) of one named stage of the last run, measured with CUDA events on the run's stream:
 * "transform_crop", "grid", "key_hist", "sort", "centroid", "total", and "sort_pass0" (the first radix pass alone; -1 when
 * the key width was decided on the device). Needs cm_set_profiling(h, 1). */
CM_API int cm_set_profiling(cm_handle_t h, int on);
CM_API int cm_stage_ms(cm_handle_t h, const char* stage, float* ms);

/* Debug only: with the environment variable CM_TRACE=1 set at creation, the transform_crop kernel (which = 0) and one
 * radix pass (which = 1, pass CM_TRACE_PASS) record 8 clock64 stamps per tile; this copies them out. */
CM_API int cm_debug_trace(cm_handle_t h, int which, uint64_t* out, int64_t capacity, int64_t* n);

/* ---- small device-memory helpers so that non-CUDA callers (ctypes, cgo, JNI) can stage data ---- */
CM_API int cm_dev_alloc(cm_handle_t h, void** p, size_t bytes);
CM_API int cm_dev_free(cm_handle_t h, void* p);
CM_API int cm_memcpy_h2d(cm_handle_t h, void* dst_dev, const void* src_host, size_t bytes, void* stream);
CM_API int cm_memcpy_d2h(cm_handle_t h, void* dst_host, const void* src_dev, size_t bytes, void* stream);
CM_API int cm_memcpy_d2d(cm_handle_t h, void* dst_dev, const void* src_dev, size_t bytes, void* stream);
/* a CUDA stream (non-blocking) for the `stream` argument of the device-resident calls: lets the per-sensor stages of
 * several sensors run concurrently from their own host threads, as the reference's callbacks do on ros::AsyncSpinner(6)
 * (pc_preprocessing_main.cpp:513). One handle must still only be used by one thread at a time. */
CM_API int cm_stream_create(cm_handle_t h, void** stream);
CM_API int cm_stream_destroy(cm_handle_t h, void* stream);
CM_API int cm_stream_sync(cm_handle_t h, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CLOUD_MERGER_GPU_H_ */
