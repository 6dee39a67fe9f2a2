// cm_common.cuh -- device-side structures and helpers shared by the sm_100a kernels of the merge hot path.
//
// Conventions
//  * one "run" = one batch of F frames x S sensors = n_seg segments, processed by a fixed sequence of launches;
//  * the streaming kernels (transform_crop, centroid, zone slicing) compact tile-locally and leave one count per tile; a
//    small scan kernel turns the counts into dense offsets, so they carry no inter-CTA dependency. Only the radix passes
//    need an order-preserving prefix across CTAs while the data moves: workers publish per-tile digit counts, scanner CTAs
//    turn them into running sums (cm_radix_sort.cu); tiles are handed out by an atomic counter, so forward progress does
//    not depend on which CTAs are resident;
//  * look-back words carry an epoch (device-resident, advanced once per run), so the arrays never need clearing;
//  * all spin loops have a watchdog: a stuck wait raises CM_E_INTERNAL in the control block instead of hanging the GPU.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#define CM_RADIX_BITS 8
#define CM_RADIX 256
#define CM_MAX_SORT_PASSES 8

#define CM_DEV_OK 0
#define CM_DEV_E_KEY_RANGE 5
#define CM_DEV_E_INTERNAL 6

namespace cm {

// ---- one sensor cloud of one frame, as the kernels see it ------------------------------------------------------
enum SegMode : uint32_t {
  SEG_PACKED16 = 0,  // point_step 16, x y z i at 0 4 8 12: one 16-byte load per point
  SEG_PCL32 = 1,     // pcl::PointXYZI / Velodyne-Melodic: point_step 32, xyz at 0 4 8, intensity at 16
  SEG_ALIGNED4 = 2,  // point_step % 4 == 0 and offsets % 4 == 0: four 4-byte loads
  SEG_STAGED = 3,    // anything else up to CM_MAX_STAGED_STEP: tile bytes staged to shared memory by cp.async.bulk
  SEG_BYTES = 4      // last resort: byte loads from global memory
};
#define CM_MAX_STAGED_STEP 96

struct SegDev {  // 128 bytes: one descriptor read per tile
  const uint8_t* data;
  uint32_t n_points;
  uint32_t tile_begin;      // first K1 tile of this segment (every segment owns >= 1 tile)
  uint32_t src_base;        // index of this segment's point 0 in its frame's un-cropped concatenation
  uint32_t slot_base;       // index of this segment's point 0 in the batch's un-cropped concatenation
  uint32_t frame;
  int32_t point_step;
  int32_t off_x, off_y, off_z, off_i;
  uint32_t is_dense;
  uint32_t sensor;
  uint32_t first_of_frame;
  uint32_t mode;
  uint32_t pad_;
  float m[12];              // the sensor's extrinsic, rows 0..2 of the 4x4, row-major
  uint32_t pad2_[3];
};
static_assert(sizeof(SegDev) == 128, "SegDev must stay 128 bytes");

struct PassDev {
  int32_t axis;
  float lo, hi;
  int32_t negative;
};

struct CropDev {
  int32_t n_pass;
  PassDev pass[8];
  // When every pass is a plain (non-negative) window with non-NaN limits the chain collapses to one box:
  // keep <=> lo[a] <= v[a] <= hi[a] for a = x, y, z (limits default to +-FLT_MAX, which also rejects non-finite
  // coordinates exactly like PassThrough does) and, if use_i, for the intensity field.
  int32_t is_box;
  int32_t use_i;
  float lo[4], hi[4];
};

// ---- pcl::CropBox stages after the PassThrough chain (cm_set_crop_boxes) ---------------------------------------------
// One stage with everything PCL derives per filter() call precomputed on the host: the three skip decisions (Eigen's fuzzy
// isIdentity / the exact zero compares) and the float inverse of the rotation. Not the collapsed axis-aligned chain
// (CropDev::is_box / BoxGrid): these boxes are oriented and may be negative.
#define CM_MAX_CROP_BOXES 8
#define OBOX_TRANSFORM 1u    // local = transform * p
#define OBOX_TRANSLATE 2u    // local -= translation
#define OBOX_ROTATE 4u       // local = inverse rotation * local
#define OBOX_NEGATIVE 8u
struct OrientedBoxDev {  // 144 bytes: nine 16-byte loads
  float t[12];           // setTransform, rows 0..2 row-major
  float r[12];           // inverse of the rotation (an Affine3f: its translation column is +-0)
  float tr[3];           // setTranslation
  float mn[3], mx[3];
  uint32_t flags;        // OBOX_*
  uint32_t pad_[2];
};
static_assert(sizeof(OrientedBoxDev) == 144, "OrientedBoxDev is loaded as 16-byte words");

// ---- zone slicing (cm_zones.cu): several PassThrough chains evaluated in one pass ---------------------------------------
#define CM_MAX_ZONES 16
#define CM_MAX_ZONE_PASSES 4
struct ZoneDev {
  int32_t n_pass;
  PassDev pass[CM_MAX_ZONE_PASSES];
  // When every stage is a plain (non-negative) window with non-NaN limits the chain is one box, like CropDev:
  // keep <=> lo[a] <= v[a] <= hi[a] for x, y, z (defaults +-FLT_MAX also reject non-finite coordinates) and, if use_i,
  // for the intensity.
  int32_t is_box, use_i;
  float lo[4], hi[4];
};
struct ZoneSet {
  int32_t n_zones;
  int32_t all_box;  // every zone has at least one stage and is a box: the kernels take the compare-only path
  ZoneDev zone[CM_MAX_ZONES];
};

// ---- one record per K1 tile: where the tile's survivors sit (tile-local compaction) and where they belong densely ----
struct TileRec {
  uint32_t count;   // survivors of this tile; they occupy slots [slot0, slot0 + count)
  uint32_t slot0;   // = position of the tile's first input point in the batch's un-cropped concatenation
  uint32_t frame;
  uint32_t dense0;  // exclusive prefix of count over all earlier tiles (filled by k_tile_scan)
};

// ---- per-run control block; zeroed by one memset at the start of every run --------------------------------------
struct FrameAcc {
  uint32_t max_enc[3];   // atomicMax of enc(v)         -> max_p
  uint32_t nmin_enc[3];  // atomicMax of ~enc(v)        -> min_p
  uint32_t n_invalid;    // survivors with a non-finite coordinate (only possible when no crop pass is configured)
  uint32_t voxel_count;  // voxels emitted for this frame
};

struct Ctrl {
  uint32_t tile_counter[12];  // [1 + p]: next tile of radix pass p (the persistent workers claim tiles here); others unused
  uint32_t error;             // CM_DEV_E_*
  uint32_t total_voxels;
  uint32_t has_invalid;
  uint32_t pad_;
  uint32_t role_counter[CM_MAX_SORT_PASSES];  // [p]: arrival ticket of the CTAs of radix pass p (the first arrivals scan)
  uint32_t cent_ticket;       // next tile of the persistent centroid kernel
  uint32_t pad2_[7];
};
static_assert(sizeof(Ctrl) == 128, "Ctrl is two cache lines");

// ---- written by k_grid_setup -----------------------------------------------------------------------------------
struct GridDev {
  int32_t min_b[3];
  int32_t max_b[3];
  int32_t div_b[3];
  int32_t pcl_overflow;
  uint32_t bits;
  uint32_t empty;
  uint32_t zero_keys;             // 1: the grid is outside the key range (or PCL refuses the frame in overflow mode 1): every
                                  // point of the frame gets voxel index 0, so no key leaves the frame's (1-cell) grid
  unsigned long long mul1, mul2;  // div0, div0*div1
};

struct SortInfo {
  uint32_t num_passes;
  uint32_t total_bits;
  uint32_t idx_bits;
  uint32_t n_keys;      // = survivors
  uint32_t key_frames;  // F (+1 when a sentinel frame is needed for invalid points)
  uint32_t width;       // bytes of the keys that travel through the sort: 4 (8-byte records) or 8
  uint32_t segmented;   // frame-segmented sort: the keys are the voxel index alone (no frame bits), every frame is sorted as its
                        // own segment of the frame-ordered input, the frame of a key is known from its position
  uint32_t n_seg_tiles; // seg_sort: number of (frame-aligned) radix tiles
  uint32_t seg_sort;    // the passes sort every frame as a segment of its own: segmented runs, and fused-key runs whose frame
                        // bits stay in the keys but are not ranked (BoxGrid::seg_sort)
};

// One radix tile of a frame-segmented sort: tiles never straddle frames.
struct SegTile {
  uint32_t base;   // position of the tile's first key (in every ping-pong buffer: a frame keeps its range)
  uint32_t n;      // keys in the tile (< tile size only for the last tile of a frame)
  uint32_t frame;  // bit 31: first tile of its frame
  uint32_t pad;
};
constexpr uint32_t CM_SEG_FIRST = 0x80000000u;
constexpr uint32_t CM_SEG_PASSES = 4;  // a segmented key is 32 bits wide at most
// Bins of a wide top digit: the last pass of a fused-key run may rank up to 384 values of the box-grid index (BoxGrid::top_bins)
// instead of 256. A frame's row of seg_hist holds it as long as it is pass 2 or earlier (2 * 256 + 384 <= 4 * 256).
constexpr uint32_t CM_WIDE_BINS = 384;

// ---- float <-> order-preserving uint -----------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t f32_order_enc(uint32_t bits) {
  return bits ^ ((bits >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__host__ __device__ __forceinline__ uint32_t f32_order_dec(uint32_t enc) {
  return enc ^ ((enc >> 31) ? 0x80000000u : 0xFFFFFFFFu);
}

#ifdef __CUDACC__

__device__ __forceinline__ bool finite_f32(float v) { return (__float_as_uint(v) & 0x7F800000u) != 0x7F800000u; }

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ uint32_t lanemask_lt() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

__device__ __forceinline__ uint32_t warp_sum_u32(uint32_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}
__device__ __forceinline__ uint32_t warp_incl_scan_u32(uint32_t v) {
  const uint32_t lane = lane_id();
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v, o);
    if (lane >= (uint32_t)o) v += t;
  }
  return v;
}

// streaming 16-byte accesses that do not pollute L1
__device__ __forceinline__ float4 ldg_stream_f4(const void* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float ldg_stream_f1(const void* p) {
  float r;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}

// ---- decoupled look-back --------------------------------------------------------------------------------------
// word = ((epoch * 4 + flag) << 32) | value ; flag 1 = tile aggregate published, 2 = inclusive prefix published.
#define CM_LB_AGG 1u
#define CM_LB_INCL 2u
#define CM_SPIN_LIMIT (1u << 22)
// Watchdog of the spin loops: wall-clock based (%globaltimer, nanoseconds), so that a kernel that merely shares the GPU
// with other work (several handles sorting at once, MPS, time slicing) is not mistaken for a stuck one. The timer is read
// once every CM_WATCHDOG_STRIDE polls.
#define CM_WATCHDOG_NS 4000000000ull
#define CM_WATCHDOG_STRIDE 1024u

__device__ __forceinline__ unsigned long long lb_pack(uint32_t epoch, uint32_t flag, uint32_t value) {
  return ((unsigned long long)(epoch * 4u + flag) << 32) | (unsigned long long)value;
}

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// Weak load served by L2 (L1 bypassed), so it observes other SMs' stores, and -- unlike the strong load above, which the
// hardware completes one at a time per thread (measured: ~300 cycles each, back to back) -- several can be in flight.
// Used for the batched window reads of the look-back; the spin on a single word keeps the strong load.
__device__ __forceinline__ unsigned long long ld_cg_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_cg_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.global.cg.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ bool lb_ready(unsigned long long w, uint32_t epoch) {
  const uint32_t hi = (uint32_t)(w >> 32);
  return (hi >> 2) == epoch && (hi & 3u) != 0u;
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// One poll of a spin loop went by without success: true once the loop has been spinning for CM_WATCHDOG_NS. `spins` and
// `t0` are the loop's own state (t0 = 0 until the first timer read).
__device__ __forceinline__ bool watchdog_expired(uint32_t& spins, unsigned long long& t0) {
  if ((++spins & (CM_WATCHDOG_STRIDE - 1u)) != 0u) return false;
  const unsigned long long now = global_timer_ns();
  if (t0 == 0ull) {
    t0 = now;
    return false;
  }
  return now - t0 > CM_WATCHDOG_NS;
}

// Spin until the word of this epoch carries the INCLUSIVE flag (written by the scanner CTAs of the radix pass).
__device__ __forceinline__ uint32_t lb_wait_inclusive(unsigned long long* p, uint32_t epoch, uint32_t* err) {
  uint32_t spins = 0;
  unsigned long long t0 = 0ull;
  while (true) {
    const unsigned long long w = ld_relaxed_u64(p);
    const uint32_t hi = (uint32_t)(w >> 32);
    if ((hi >> 2) == epoch && (hi & 3u) == CM_LB_INCL) return (uint32_t)w;
    if (watchdog_expired(spins, t0)) {
      atomicExch(err, (uint32_t)CM_DEV_E_INTERNAL);
      return 0u;
    }
    if (spins > 16) __nanosleep(40);
  }
}

// Exclusive scan over 256 values held one per thread by threads 0..255 of a block with >= 256 threads.
// `scratch` is >= 9 uint32 of shared memory. Every thread of the block must call it; returns the exclusive prefix
// (for threads >= 256 the return value is meaningless). *total receives the sum (valid in all threads).
// Exclusive scan of one value per thread over the first N threads of the block (N / 32 warps; scratch >= N / 32 + 1 words).
template <int N>
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* scratch, uint32_t* total) {
  constexpr int W = N / 32;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
  if (tid >= (uint32_t)N) v = 0;
  const uint32_t incl = warp_incl_scan_u32(v);
  if (lane == 31 && w < W) scratch[w] = incl;
  __syncthreads();
  if (tid == 0) {
    uint32_t run = 0;
#pragma unroll
    for (int i = 0; i < W; ++i) {
      uint32_t t = scratch[i];
      scratch[i] = run;
      run += t;
    }
    scratch[W] = run;
  }
  __syncthreads();
  const uint32_t res = incl - v + (w < W ? scratch[w] : 0u);
  *total = scratch[W];
  __syncthreads();
  return res;
}
__device__ __forceinline__ uint32_t block_excl_scan_256(uint32_t v, uint32_t* scratch, uint32_t* total) {
  return block_excl_scan<256>(v, scratch, total);
}

#endif  // __CUDACC__

}  // namespace cm
