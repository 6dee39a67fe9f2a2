// cm_kernels.h -- launch interface between the C-ABI host layer (cm_api.cu) and the sm_100a kernels.
#pragma once

#include <algorithm>

#include "cm_common.cuh"

namespace cm {

// ---- K1: fused unpack + transform + crop + stable compaction (cm_transform_crop.cu) ---------------------------------
#define K1_BIG_BATCH_POINTS (1u << 21)
// Voxel keys straight out of K1 (round 2). When the crop chain is a box that bounds x, y and z, the voxel grid of that BOX
// contains the grid PCL derives from the data of any frame, and ordering by (k, j, i) does not depend on the grid origin:
// K1 can key every survivor against the box grid the moment it is transformed, and count the digits of every radix pass
// while it is at it. That removes k_voxel_key_hist (a 16-byte re-read of every survivor plus a launch). The key of a
// survivor is written at its slot (4 bytes; the slot is the read position, so no value travels), radix pass 0 reads the
// keys tile-locally through the K1 tile records, and k_voxel_centroid turns the box-grid index of a voxel back into PCL's
// idx = i + j*div_x + k*div_x*div_y on the frame's data-derived grid.
struct BoxGrid {
  float inv[3];              // inverse leaf
  int32_t min_b[3];          // floor(box_lo * inv)
  uint32_t mul1, mul2;       // div_x, div_x * div_y of the box grid
  uint32_t idx_bits;         // bits of the largest box-grid index: key = (frame << idx_bits) | idx
  uint32_t n_pass;           // radix passes the run will make
};
struct K1Params {
  const SegDev* segs;
  uint32_t n_seg;
  uint32_t n_tiles;
  uint32_t n_frames;
  uint32_t tiles_per_seg;    // > 0: every segment owns exactly this many tiles (segment = tile / tiles_per_seg)
  const uint32_t* tile_seg;  // otherwise: segment of every tile
  CropDev crop;
  float4* surv_xyzi;
  uint32_t* surv_src;  // may be null
  Ctrl* ctrl;
  FrameAcc* acc;
  uint32_t* surv_key;          // [slots] box-grid voxel key of every survivor, or null: keys come from k_voxel_key_hist
  uint32_t* hist;              // [CM_MAX_SORT_PASSES][256] digit histograms of all passes (with surv_key)
  BoxGrid box;
  TileRec* tile_rec;           // [n_tiles] out: count / slot0 / frame of every tile
  unsigned long long* trace;   // debug: 8 clock64 stamps per tile, or null
};
uint32_t k1_tile_points(int64_t total_points);
uint32_t k1_min_tile_points();
uint32_t k1_staged_smem(uint32_t tile_points, uint32_t max_step);
// mode: SEG_PACKED16 / SEG_PCL32 when every segment of the launch has that layout, anything else = generic kernel
cudaError_t launch_transform_crop(const K1Params& p, uint32_t tile_points, int mode, uint32_t staged_smem_bytes,
                                  cudaStream_t stream);

// One CTA: exclusive prefix of TileRec.count -> TileRec.dense0, frame_surv_start[f] (first tile of each frame),
// frame_surv_start[n_frames] = total, seg_surv_start[s].
cudaError_t launch_tile_scan(TileRec* tile_rec, uint32_t n_tiles, const SegDev* segs, uint32_t n_seg, uint32_t n_frames,
                             uint32_t* frame_surv_start, uint32_t* seg_surv_start, cudaStream_t stream);
// Dense copy of the merged cropped cloud (xyzi + source index + slot of every survivor), on request only.
cudaError_t launch_compact_survivors(const TileRec* tile_rec, uint32_t n_tiles, const float4* slot_xyzi,
                                     const uint32_t* slot_src, float4* dense_xyzi, uint32_t* dense_src,
                                     uint32_t* dense_slot, cudaStream_t stream);

// ---- VoxelGrid front/back ends (cm_voxel.cu) ---------------------------------------------------------------------
struct VoxelParams {
  const float4* pts;                 // survivors by slot (tile-locally compacted), or a plain dense cloud
  const TileRec* tile_rec;           // K1's tile records; null = pts is dense (slot == index, one frame)
  uint32_t n_k1_tiles;
  const uint32_t* frame_surv_start;  // [n_frames + 1]; [n_frames] = number of points M
  uint32_t n_frames;
  uint32_t max_points;               // host-side upper bound of M (sizes the grids)
  float inv_leaf[3];
  uint32_t min_points;
  uint32_t downsample_all;
  uint32_t pcl_refuses;              // overflow mode 1: a frame PCL refuses is returned as its cropped cloud, so a grid of that
                                     // frame beyond the key range is not an error
  uint32_t key_bytes;                // 4 or 8
  uint32_t out_step;                 // 16 or 32
  Ctrl* ctrl;
  FrameAcc* acc;
  GridDev* grid;                     // [n_frames]
  SortInfo* info;
  uint32_t* hist;                    // [CM_MAX_SORT_PASSES][256]
  void* keys_a;                      // ping-pong: 64-bit keys, or 8-byte (key, value) records when key_bytes == 4
  void* keys_b;
  uint32_t* vals_a;                  // values of 64-bit keys (unused by the record layout)
  uint32_t* vals_b;
  unsigned long long* lb_sort;       // [sort tiles][256]
  unsigned long long* cent_status;   // [centroid tiles] look-back words of the voxel compaction (epoch-tagged, never cleared)
  uint32_t cent_status_words;
  uint32_t* epoch_dev;               // device-resident run epoch: advanced by 16 in k_grid_setup, read by the sort passes
                                     // (pass p tags its look-back words with *epoch_dev + 1 + p), so no kernel argument
                                     // changes from run to run and a captured launch sequence can be replayed as a graph
  uint32_t lb_sort_words;            // size of lb_sort, for the clear on epoch wrap-around
  uint32_t max_passes;               // how many pass launches the host enqueues
  uint32_t fused_keys;               // K1 already wrote the (box-grid) keys at the survivors' slots and counted the digits:
                                     // no k_voxel_key_hist; radix pass 0 reads surv_key through the K1 tile records
  const uint32_t* surv_key;          // [slots]
  BoxGrid box;
  uint32_t* first_k1;                // [sort tiles] K1 tile that holds dense position t * sort_tile (written by k_grid_setup)
  uint32_t sort_tile;                // keys per tile of the radix passes of this run
  uint32_t dual_width;               // the key width is only known on the device (SortInfo.width): the host enqueues the
                                     // 32-bit AND the 64-bit instantiation of every kernel, the one that does not apply exits
  // Frame-segmented sort (batches of several frames): the frame bits are not sorted -- the input is frame-ordered already --
  // so the keys are the bare voxel index: 32-bit records where (frame, index) needed 64 bits, and fewer passes.
  uint32_t segmented;                // 0: never; 1: the device decides (dual_width runs: segmented 32-bit or plain 64-bit);
                                     // 2: the host decided (bounded grid)
  SegTile* seg_tile;                 // [sort tiles + frames] written by k_grid_setup
  uint32_t* seg_hist;                // [n_frames][CM_SEG_PASSES][256] digit counts per frame, turned into first positions
                                     // (frame start + exclusive scan) by k_seg_base
  uint32_t* seg_frame_tile0;         // [n_frames + 1] scratch of k_grid_setup
  uint2* seg_cent_range;             // [centroid tiles] first and last frame with items in the tile (k_grid_setup)
  void* out_xyzi;
  uint32_t* out_count;
  unsigned long long* out_idx;
  unsigned long long* trace;         // debug: 8 clock64 stamps per tile of the traced kernel, or null
  uint32_t trace_pass;               // which sort pass writes the trace
};

// bounding box of n packed points (used when VoxelGrid runs on a cloud that did not come out of K1)
cudaError_t launch_minmax(const float4* pts, uint32_t n, Ctrl* ctrl, FrameAcc* acc, uint32_t* frame_surv_start,
                          cudaStream_t stream);
cudaError_t launch_seed_bounds(FrameAcc* acc, const float* mn, const float* mx, cudaStream_t stream);
// one CTA; when scan_rec is given it first does launch_tile_scan's work (K1 tile counts -> dense offsets, frame / segment starts)
cudaError_t launch_grid_setup(const VoxelParams& p, cudaStream_t stream, TileRec* scan_rec = nullptr, uint32_t scan_tiles = 0,
                              const SegDev* segs = nullptr, uint32_t n_seg = 0, uint32_t* seg_surv_start = nullptr);
cudaError_t launch_key_hist(const VoxelParams& p, cudaStream_t stream);
cudaError_t launch_seg_base(const VoxelParams& p, cudaStream_t stream);  // segmented runs: between key_hist and the passes
// segmented runs sort bare voxel indices; this hands out (frame << idx_bits | idx) keys and the values as two arrays
cudaError_t launch_seg_keys64(const void* records, unsigned long long* keys, uint32_t* vals, const VoxelParams& p,
                              cudaStream_t stream);
cudaError_t launch_sort_pass(const VoxelParams& p, int pass, cudaStream_t stream);
// 32-bit keys are sorted as 8-byte (key, value) records in keys_a/keys_b; this splits the first *n_ptr records into two arrays
// remap != null (fused-key run): the keys index the crop box's grid; they are handed out re-based on each frame's data-derived
// grid (PCL's idx), frame bits kept
cudaError_t launch_split_records(const void* records, uint32_t* keys, uint32_t* vals, const uint32_t* n_ptr,
                                 uint32_t max_points, cudaStream_t stream, const VoxelParams* remap = nullptr);
cudaError_t launch_centroid(const VoxelParams& p, cudaStream_t stream);        // one launch: runs, centroids, dense ordered output
#define CM_CENTROID_LAUNCHES 1
// host path: dense voxel outputs of a one-frame run -> device-mapped page-locked host arrays, sized by Ctrl.total_voxels
cudaError_t launch_export_voxels(const VoxelParams& p, void* host_xyzi, uint32_t* host_count, unsigned long long* host_idx,
                                 uint32_t cap, cudaStream_t stream);

// ---- zone slicing: multi-output PassThrough compaction (cm_zones.cu) -------------------------------------------------------
struct GiantPlan;
struct ZoneParams {
  const float4* pts;         // n packed xyzi points
  uint32_t n_points;
  uint32_t n_tiles;          // ceil(n_points / zone_tile_points())
  ZoneSet zones;
  unsigned short* mask;      // [n_points] zone membership of every point
  uint32_t mask_given;       // the masks were produced by another kernel (radius outlier removal): only count them
  uint32_t* tile_count;      // [n_zones][n_tiles]
  uint32_t* tile_offset;     // [n_zones][n_tiles] where the tile's points of the zone start, relative to the zone's start
  uint32_t* zone_total;      // [n_zones] points per zone
  uint32_t* scan_ticket;     // counts the zone CTAs of k_zone_scan that have finished (self-resetting)
  uint32_t* zone_begin;      // [n_zones + 1] zone z occupies [zone_begin[z], zone_begin[z+1]) of the output
  uint32_t* overflow;        // set to the needed size when the zones together exceed out_capacity
  uint32_t out_capacity;
  float4* out_xyzi;
  uint32_t* out_src;         // index of every output point in the input cloud
  // giant-cloud exchange fused into the scatter (cm_giant_voxelgrid over peer memory): zone r is written straight into rank
  // r's receive buffer (an IPC-mapped pointer; NVLink stores), from element zone_remote_base[r] on; no source indices
  float4* zone_ptr[CM_MAX_ZONES];        // all null: the ordinary local outputs
  const uint32_t* zone_remote_base;      // [n_zones], device
  // giant-cloud mode: the "zone" of a point is the rank that owns its voxel index (device-resident plan: global grid and
  // splitters); the count kernel derives the masks from it in the same sweep (mask_given must be 0)
  const GiantPlan* giant_plan;           // null: zones / given masks
  uint32_t giant_invalid_part;           // where non-finite points go (the local rank)
};
// ---- radius outlier removal on the sorted cell keys (cm_outlier.cu) -------------------------------------------------------
struct RorParams {
  float r2;              // (float)(radius * radius): FLANN counts squared distances strictly below it
  uint32_t min_pts;      // keep iff count (the point itself included) > min_pts
  uint32_t negative;
  unsigned short* mask;  // [n_points] keep flag per input point (cleared by the caller)
  uint32_t* cell_start;  // [table_keys + 1] first sorted position with key >= k, or nullptr: binary searches instead
  uint32_t table_keys;   // n_frames << idx_bits: every valid key is below it
};
// fills cell_start from the sorted keys (one launch), then counts (one launch)
cudaError_t launch_radius_table(const VoxelParams& p, const RorParams& r, cudaStream_t stream);
cudaError_t launch_radius_count(const VoxelParams& p, const RorParams& r, cudaStream_t stream);

// ---- RANSAC ground plane (cm_plane.cu) --------------------------------------------------------------------------------------
#define CM_MAX_PLANE_CLOUDS (CM_MAX_ZONES / 2)
struct PlaneParams {  // one batch of draws for up to CM_MAX_PLANE_CLOUDS independent clouds
  const float4* pts;                         // the clouds, one after the other
  uint32_t n_clouds;
  uint32_t begin[CM_MAX_PLANE_CLOUDS + 1];   // cloud k = pts[begin[k] .. begin[k+1])
  uint32_t n_draws[CM_MAX_PLANE_CLOUDS];     // draws of cloud k in this batch (0: the cloud is finished)
  uint32_t draw_stride;                      // per-draw arrays: cloud k owns [k * draw_stride, (k+1) * draw_stride)
  float threshold;         // smallest float >= the double threshold: |d| < threshold decides like PCL's float-vs-double test
  uint32_t sum_order;      // order of Eigen's 4-wide reductions: 0 SSE2 (l0+l2)+(l1+l3), 1 SSE3 (l0+l1)+(l2+l3), 2 scalar
  const int32_t* samples;  // [draw][3] point indices (relative to the cloud's first point)
  float4* models;          // [draw] plane of every draw
  int32_t* counts;         // [draw] inliers of every draw (cleared by the caller)
  int32_t* good;           // [draw] isSampleGood
};
struct PlaneSelect {
  const float4* pts;
  uint32_t n_clouds;
  uint32_t begin[CM_MAX_PLANE_CLOUDS + 1];
  uint32_t found[CM_MAX_PLANE_CLOUDS];       // 0: segment() failed for this cloud, no inliers
  float4 coeff[CM_MAX_PLANE_CLOUDS];
  float threshold;
  unsigned short* mask;    // bit 2k: inlier of cloud k, bit 2k + 1: its other points
};
cudaError_t launch_plane_score(const PlaneParams& p, cudaStream_t stream);
cudaError_t launch_plane_select(const PlaneSelect& q, uint32_t sum_order, cudaStream_t stream);
// PCL-order float sums xx xy xz yy yz zz x y z over the inliers of every cloud's model (index order) ->
// out[16 k + 0..8], out[16 k + 9] = the inlier count's bits
cudaError_t launch_plane_moments(const PlaneSelect& q, uint32_t sum_order, float* out, cudaStream_t stream);

// ---- giant-cloud mode: routing by voxel-key range (cm_route.cu) ----------------------------------------------------------
struct RouteGrid {  // PCL's grid on the GLOBAL bounding box
  float inv[3];
  long long min_b[3];
  long long div0, div01;  // div_x, div_x * div_y
};
#ifdef __CUDACC__
// PCL's voxel index of a point on the global grid (VoxelGrid::applyFilter, float32 multiply); false: a non-finite point
__device__ __forceinline__ bool route_key(const RouteGrid& g, const float4& v, unsigned long long* key) {
  if (!(finite_f32(v.x) && finite_f32(v.y) && finite_f32(v.z))) return false;
  const long long i0 = (long long)__float2int_rd(__fmul_rn(v.x, g.inv[0])) - g.min_b[0];
  const long long i1 = (long long)__float2int_rd(__fmul_rn(v.y, g.inv[1])) - g.min_b[1];
  const long long i2 = (long long)__float2int_rd(__fmul_rn(v.z, g.inv[2])) - g.min_b[2];
  *key = (unsigned long long)(i0 + i1 * g.div0 + i2 * g.div01);
  return true;
}
#endif
struct RouteSplit {
  int32_t n_parts;                           // <= CM_MAX_ZONES
  uint32_t invalid_part;                     // where non-finite points go (the local rank)
  unsigned long long splitter[CM_MAX_ZONES];  // part r owns voxel indices in [splitter[r-1], splitter[r])
};
cudaError_t launch_route_hist(const float4* pts, uint32_t n, const RouteGrid& g, unsigned long long width, uint32_t bins,
                              unsigned long long* hist, cudaStream_t stream);
cudaError_t launch_route_mask(const float4* pts, uint32_t n, const RouteGrid& g, const RouteSplit& sp, unsigned short* mask,
                              cudaStream_t stream);
// Device-resident plan of one giant-cloud run (cm_giant_voxelgrid): everything the routing kernels need comes from device
// memory, so no step of the partition waits for the host.
struct GiantPlan {
  RouteGrid grid;                               // PCL's grid on the all-reduced bounding box
  unsigned long long width;                     // voxel indices per histogram bin
  unsigned long long cells;                     // div_x * div_y * div_z
  unsigned long long total;                     // finite points of the whole cloud (sum of the all-reduced histogram)
  unsigned long long splitter[CM_MAX_ZONES];    // rank r owns voxel indices in [splitter[r-1], splitter[r])
  uint32_t enc[6];                              // the all-reduced bounds as FrameAcc holds them: max_enc[3], nmin_enc[3]
  int32_t min_b[3], div_b[3];
  uint32_t key_bits;                            // bits of the largest voxel index
  uint32_t error;                               // CM_DEV_E_KEY_RANGE: grid outside the key range
  uint32_t n_invalid;                           // THIS rank's non-finite points (not all-reduced): they stay on this rank
};
cudaError_t launch_giant_plan(GiantPlan* plan, const FrameAcc* acc_reduced, const float* inv_leaf3, uint32_t bins, cudaStream_t stream);
cudaError_t launch_giant_hist(const float4* pts, uint32_t n, const GiantPlan* plan, uint32_t bins, unsigned long long* hist,
                              cudaStream_t stream);
cudaError_t launch_giant_splitters(GiantPlan* plan, const unsigned long long* hist_reduced, uint32_t bins, uint32_t n_parts,
                                   cudaStream_t stream);
// folds device-resident bounds (GiantPlan::enc) into frame 0's accumulator: every rank then builds the same grid
cudaError_t launch_seed_bounds_enc(FrameAcc* acc, const uint32_t* enc6, cudaStream_t stream);
// bounding box of n packed points into acc (frame 0), as launch_minmax does for the VoxelGrid-only entry
uint32_t zone_tile_points();
cudaError_t launch_zone_count_scan(const ZoneParams& p, cudaStream_t stream);      // the first two launches of a split
cudaError_t launch_zone_scatter_remote(const ZoneParams& p, cudaStream_t stream);  // the third, into zone_ptr[] (peer memory)
// where this rank's part of every destination starts in that destination's receive buffer, from the all-gathered offsets
// (row s = rank s's zone_begin[0 .. world], entry CM_MAX_ZONES + 1 = its receive capacity); *overflow != 0: some rank would
// receive more than it can hold (every rank sees the same) and nobody writes
cudaError_t launch_giant_offsets(const uint32_t* counts_all, uint32_t stride, uint32_t world, uint32_t me, uint32_t* remote_base,
                                 uint32_t* overflow, cudaStream_t stream);
cudaError_t launch_zone_split(const ZoneParams& p, cudaStream_t stream);  // 3 launches
cudaError_t launch_zone_scatter(const ZoneParams& p, cudaStream_t stream);  // the last of them again, after out_* grew
#define CM_ZONE_LAUNCHES 3

uint32_t sort_tile_items(uint32_t key_bytes, uint32_t max_points);
size_t sort_lookback_rows(uint32_t capacity);
uint32_t centroid_tile_items();

// per-device one-time kernel attribute setup (opt-in shared memory sizes)
cudaError_t configure_device_kernels();
cudaError_t configure_sort_kernels();

}  // namespace cm
