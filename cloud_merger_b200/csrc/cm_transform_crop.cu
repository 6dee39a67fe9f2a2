// cm_transform_crop.cu -- K1: fused PointCloud2 unpack + rigid transform + PassThrough crop + stable stream compaction
// (+ per-frame bounding box of the survivors) for sm_100a.
//
// Replaces, in one pass over the raw bytes (reference paths relative to timspilak/cloud_merger):
//   * the pcl_ros subscriber deserialisation            pc_preprocessing_main.cpp:520-525
//   * pcl_ros::transformPointCloud                      pc_preprocessing_main.cpp:322,348,373,399,426,465
//   * the pcl::PassThrough chains getROI/getCloudPart   pc_preprocessing_main.cpp:20-59 (and CloudFusionNode.h:145-216)
//   * the operator+= concatenation in fusePointclouds   pc_preprocessing_main.cpp:137-149
//   * pcl::CropBox stages after the chain (vehicle body) (PCL 1.8.1 crop_box.hpp; cm_set_crop_boxes)
//   * pcl::getMinMax3D, the first step of VoxelGrid     (PCL 1.8.1 voxel_grid.hpp)
//
// Roofline: HBM. Algorithmic bytes per launch = sum(n_points * point_step) + survivors * (16 + 4).
// Arithmetic is kept bit-identical to the PCL 1.8.1 CPU build: x' = ((m00*x + m01*y) + m02*z) + m03 with every
// multiply and add rounded separately (__fmul_rn/__fadd_rn are never contracted into FMA).
//
// Structure: one tile per CTA and no dependency between CTAs: a tile compacts its survivors, in input order, to the
// head of its own slot range [slot0, slot0 + count) and leaves a 16-byte TileRec; the one-CTA k_tile_scan then turns the
// counts into dense offsets (frame starts, totals), and the VoxelGrid kernels address survivors by slot. A dense copy of
// the merged cloud is produced by k_compact_survivors only when a caller asks for it. The kernel is specialised at
// compile time on the record layout (16-byte packed, 32-byte PCL, generic) and on the crop kind (one
// box vs. a general chain) and on whether CropBox stages follow (OBOX; without them the kernels are what they were before
// those stages existed), which keeps the per-point instruction count low enough to stay memory-bound.
#include <cstdlib>

#include "cm_kernels.h"

namespace cm {

namespace {

constexpr int MODE_GENERIC = -1;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// 1-D TMA bulk copy global -> shared, completion signalled on the mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

__device__ __forceinline__ float lds_f32_unaligned(const uint8_t* s, uint32_t byte_off) {
  const uint32_t a = byte_off & ~3u, sh = (byte_off & 3u) * 8u;
  const uint32_t w0 = *reinterpret_cast<const uint32_t*>(s + a);
  const uint32_t w1 = *reinterpret_cast<const uint32_t*>(s + a + 4);
  return __uint_as_float(__funnelshift_r(w0, w1, sh));
}
__device__ __forceinline__ float ldg_f32_bytes(const uint8_t* p) {
  const uint32_t v = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
  return __uint_as_float(v);
}

// One pcl::PassThrough stage on a point whose x, y, z are finite (PCL 1.8.1 applyFilterIndices).
__device__ __forceinline__ bool pass_keeps(const PassDev& ps, float x, float y, float z, float it) {
  const float v = ps.axis == 0 ? x : (ps.axis == 1 ? y : (ps.axis == 2 ? z : it));
  if (!finite_f32(v)) return false;
  if (!ps.negative) return !(v < ps.lo || v > ps.hi);
  return !(v >= ps.lo && v <= ps.hi);
}

// One row of pcl::transformPoint: ((m0*x + m1*y) + m2*z) + m3, every operation rounded on its own.
__device__ __forceinline__ float affine_row(const float* m, float x, float y, float z) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], x), __fmul_rn(m[1], y)), __fmul_rn(m[2], z)), m[3]);
}

// One pcl::CropBox stage (PCL 1.8.1 CropBox::applyFilter) on a point that reached it; true = kept. The three steps are
// applied one after another, as PCL does: composing them into one matrix would round differently.
__device__ __forceinline__ bool obox_keeps(const OrientedBoxDev& b, float x, float y, float z) {
  const uint32_t f = b.flags;
  if (f & OBOX_TRANSFORM) {
    const float u = affine_row(b.t, x, y, z), v = affine_row(b.t + 4, x, y, z), w = affine_row(b.t + 8, x, y, z);
    x = u; y = v; z = w;
  }
  if (f & OBOX_TRANSLATE) {
    x = __fsub_rn(x, b.tr[0]); y = __fsub_rn(y, b.tr[1]); z = __fsub_rn(z, b.tr[2]);
  }
  if (f & OBOX_ROTATE) {
    const float u = affine_row(b.r, x, y, z), v = affine_row(b.r + 4, x, y, z), w = affine_row(b.r + 8, x, y, z);
    x = u; y = v; z = w;
  }
  // a NaN coordinate fails every compare: it counts as inside
  const bool outside = (x < b.mn[0]) | (y < b.mn[1]) | (z < b.mn[2]) | (x > b.mx[0]) | (y > b.mx[1]) | (z > b.mx[2]);
  return outside == ((f & OBOX_NEGATIVE) != 0u);
}

// BOX: 0 = general PassThrough chain, 1 = one x/y/z box, 2 = box that also windows the intensity
// min/max folded only when `on` (predicated instructions, no branch, no select)
__device__ __forceinline__ void minmax_if(bool on, float v, float& mn, float& mx) {
  asm("{\n .reg .pred p;\n setp.ne.s32 p, %2, 0;\n @p min.f32 %0, %0, %3;\n @p max.f32 %1, %1, %3;\n}"
      : "+f"(mn), "+f"(mx)
      : "r"((int)on), "f"(v));
}

template <int THREADS, int IPT, int MODE, int BOX, bool KEYS, bool OBOX>
__global__ void __launch_bounds__(THREADS, (THREADS >= 512 ? 2 : 4)) k_transform_crop(const K1Params p) {
  constexpr int TILE = THREADS * IPT;
  constexpr int WARPS = THREADS / 32;
  static_assert(!KEYS || BOX != 0, "keys are emitted against the crop box");
  extern __shared__ __align__(16) uint8_t stage[];
  // digit counts of this tile's survivors for radix pass 0 (pass 0 itself counts the digits of the later passes: K1 runs
  // one CTA per tile, and four histograms per CTA were 5 M global reductions per batch -- measured +34 us on the kernel)
  __shared__ uint32_t s_hist[KEYS ? CM_RADIX : 1];
  __shared__ uint32_t s_warp_tot[WARPS], s_warp_inv[WARPS];
  __shared__ uint32_t s_mm[WARPS][6];  // order-preserving encodings: ~enc(min) x3, enc(max) x3
  __shared__ __align__(8) unsigned long long s_bar;

  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t tile = blockIdx.x;
  const long long tr0 = clock64();
  if (KEYS && tid < CM_RADIX) s_hist[tid] = 0u;  // ordered by the barrier further down
#define K1_TRACE(i) do { if (p.trace && tid == 0) p.trace[(size_t)tile * 8 + (i)] = (unsigned long long)(clock64() - tr0); } while (0)
  // CropBox stages: the table goes to shared memory once per CTA in 16-byte words (ordered by the barrier after the unpack)
  const OrientedBoxDev* sbox = nullptr;
  uint32_t n_obox = 0;
  if constexpr (OBOX) {
    __shared__ __align__(16) OrientedBoxDev s_obox[CM_MAX_CROP_BOXES];
    n_obox = p.n_obox;
    const uint4* src = reinterpret_cast<const uint4*>(p.obox);
    for (uint32_t k = tid; k < n_obox * (uint32_t)(sizeof(OrientedBoxDev) / 16); k += THREADS)
      reinterpret_cast<uint4*>(s_obox)[k] = __ldg(src + k);
    sbox = s_obox;
  }

  // which segment owns this tile: uniform batches by division, others through the host-built table
  const uint32_t seg_id = p.tiles_per_seg ? (tile / p.tiles_per_seg) : __ldg(p.tile_seg + tile);
  const SegDev* __restrict__ sg = p.segs + seg_id;  // one 128-byte line: the first touch brings all of it
  const uint8_t* data = sg->data;
  const uint32_t seg_points = sg->n_points, tile_begin = sg->tile_begin;
  const uint32_t pt0 = (tile - tile_begin) * TILE;
  const uint32_t n_here = seg_points > pt0 ? min((uint32_t)TILE, seg_points - pt0) : 0u;

  float x[IPT], y[IPT], z[IPT], it[IPT];
  const uint32_t li0 = warp * (32 * IPT) + lane;  // local index of item 0; item i is li0 + 32*i

  // ---- unpack -------------------------------------------------------------------------------------------------
  const bool full = n_here == (uint32_t)TILE;
  if (MODE == (int)SEG_PACKED16) {
    const uint8_t* base = data + ((size_t)pt0 + li0) * 16;
    if (full) {  // no bounds checks: eight independent 16-byte loads at constant offsets
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        const float4 v = ldg_stream_f4(base + (size_t)i * (32 * 16));
        x[i] = v.x; y[i] = v.y; z[i] = v.z; it[i] = v.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (li0 + 32 * i < n_here) v = ldg_stream_f4(base + (size_t)i * (32 * 16));
        x[i] = v.x; y[i] = v.y; z[i] = v.z; it[i] = v.w;
      }
    }
  } else if (MODE == (int)SEG_PCL32) {
    const uint8_t* base = data + ((size_t)pt0 + li0) * 32;
    if (full) {
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        const float4 v = ldg_stream_f4(base + (size_t)i * (32 * 32));
        const float w = ldg_stream_f1(base + (size_t)i * (32 * 32) + 16);
        x[i] = v.x; y[i] = v.y; z[i] = v.z; it[i] = w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        float w = 0.f;
        if (li0 + 32 * i < n_here) {
          v = ldg_stream_f4(base + (size_t)i * (32 * 32));
          w = ldg_stream_f1(base + (size_t)i * (32 * 32) + 16);
        }
        x[i] = v.x; y[i] = v.y; z[i] = v.z; it[i] = w;
      }
    }
  } else {
    const uint32_t mode = sg->mode;
    const int step = sg->point_step, ox = sg->off_x, oy = sg->off_y, oz = sg->off_z, oi = sg->off_i;
    const uint8_t* base = data + (size_t)pt0 * step;
    if (mode == SEG_PACKED16) {
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        const uint32_t li = li0 + 32 * i;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (li < n_here) v = ldg_stream_f4(base + (size_t)li * 16);
        x[i] = v.x; y[i] = v.y; z[i] = v.z; it[i] = v.w;
      }
    } else if (mode == SEG_PCL32) {
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        const uint32_t li = li0 + 32 * i;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        float w = 0.f;
        if (li < n_here) {
          v = ldg_stream_f4(base + (size_t)li * 32);
          w = ldg_stream_f1(base + (size_t)li * 32 + 16);
        }
        x[i] = v.x; y[i] = v.y; z[i] = v.z; it[i] = w;
      }
    } else if (mode == SEG_ALIGNED4) {
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        const uint32_t li = li0 + 32 * i;
        x[i] = y[i] = z[i] = it[i] = 0.f;
        if (li < n_here) {
          const uint8_t* r = base + (size_t)li * step;
          x[i] = ldg_stream_f1(r + ox);
          y[i] = ldg_stream_f1(r + oy);
          z[i] = ldg_stream_f1(r + oz);
          if (oi >= 0) it[i] = ldg_stream_f1(r + oi);
        }
      }
    } else if (mode == SEG_STAGED) {
      // raw tile bytes -> shared memory with one TMA bulk copy (16-byte multiple) + a < 16-byte tail by plain loads
      const uint32_t bytes = n_here * (uint32_t)step;
      const uint32_t bulk = bytes & ~15u;
      if (tid == 0) mbar_init(&s_bar, 1);
      __syncthreads();
      if (tid == 0 && bulk) {
        mbar_arrive_expect_tx(&s_bar, bulk);
        bulk_g2s(stage, base, bulk, &s_bar);
      }
      for (uint32_t b = bulk + tid; b < bytes; b += THREADS) stage[b] = base[b];
      if (bulk) {
        uint32_t spins = 0;
        while (!mbar_try_wait(&s_bar, 0)) {
          if (++spins > CM_SPIN_LIMIT) {
            atomicExch(&p.ctrl->error, (uint32_t)CM_DEV_E_INTERNAL);
            break;
          }
        }
      }
      __syncthreads();
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        const uint32_t li = li0 + 32 * i;
        x[i] = y[i] = z[i] = it[i] = 0.f;
        if (li < n_here) {
          const uint32_t r = li * (uint32_t)step;
          x[i] = lds_f32_unaligned(stage, r + ox);
          y[i] = lds_f32_unaligned(stage, r + oy);
          z[i] = lds_f32_unaligned(stage, r + oz);
          if (oi >= 0) it[i] = lds_f32_unaligned(stage, r + oi);
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        const uint32_t li = li0 + 32 * i;
        x[i] = y[i] = z[i] = it[i] = 0.f;
        if (li < n_here) {
          const uint8_t* r = base + (size_t)li * step;
          x[i] = ldg_f32_bytes(r + ox);
          y[i] = ldg_f32_bytes(r + oy);
          z[i] = ldg_f32_bytes(r + oz);
          if (oi >= 0) it[i] = ldg_f32_bytes(r + oi);
        }
      }
    }
  }
  K1_TRACE(0);
  if (OBOX) __syncthreads();

  float m[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) m[k] = sg->m[k];
  const bool dense = sg->is_dense != 0;

  // ---- transform + crop predicate + in-warp ranks ------------------------------------------------------------------
  // Branch-free per item: the bounding box is folded with predicated min/max, the box test is one predicate chain.
  uint32_t keep_bits = 0;   // bit i: item i survives
  uint32_t ballots[IPT];    // warp-uniform
  uint32_t inv_run = 0;
  float mn0 = 3.402823466e+38f, mn1 = mn0, mn2 = mn0, mx0 = -mn0, mx1 = -mn0, mx2 = -mn0;
  const float lo0 = p.crop.lo[0], lo1 = p.crop.lo[1], lo2 = p.crop.lo[2], lo3 = p.crop.lo[3];
  const float hi0 = p.crop.hi[0], hi1 = p.crop.hi[1], hi2 = p.crop.hi[2], hi3 = p.crop.hi[3];
#pragma unroll
  for (int i = 0; i < IPT; ++i) {
    const bool in_range = full || (li0 + 32 * i < n_here);
    const float a = x[i], b = y[i], c = z[i];
    bool keep, fold;
    if (BOX) {
      // a non-finite input coordinate makes every output row non-finite, and the box rejects those, so the
      // "leave invalid points of a non-dense cloud untransformed" rule needs no special case here
      x[i] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], a), __fmul_rn(m[1], b)), __fmul_rn(m[2], c)), m[3]);
      y[i] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[4], a), __fmul_rn(m[5], b)), __fmul_rn(m[6], c)), m[7]);
      z[i] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[8], a), __fmul_rn(m[9], b)), __fmul_rn(m[10], c)), m[11]);
      keep = in_range & (x[i] >= lo0) & (x[i] <= hi0) & (y[i] >= lo1) & (y[i] <= hi1) & (z[i] >= lo2) & (z[i] <= hi2);
      if (BOX == 2) keep = keep & (it[i] >= lo3) & (it[i] <= hi3);
      // CropBox stages: their input is dense (PassThrough output) and every survivor of the box is finite; a warp whose
      // item the box already rejected everywhere skips them
      if (OBOX && __any_sync(0xFFFFFFFFu, keep))
        for (uint32_t k = 0; k < n_obox; ++k) keep = keep & obox_keeps(sbox[k], x[i], y[i], z[i]);
      fold = keep;
    } else {
      const bool fin_in = finite_f32(a) && finite_f32(b) && finite_f32(c);
      if (dense || fin_in) {
        x[i] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], a), __fmul_rn(m[1], b)), __fmul_rn(m[2], c)), m[3]);
        y[i] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[4], a), __fmul_rn(m[5], b)), __fmul_rn(m[6], c)), m[7]);
        z[i] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[8], a), __fmul_rn(m[9], b)), __fmul_rn(m[10], c)), m[11]);
      }
      const bool fin = finite_f32(x[i]) && finite_f32(y[i]) && finite_f32(z[i]);
      keep = in_range;
      const int n_pass = p.crop.n_pass;
      if (n_pass > 0) {
        keep = keep && fin;
        for (int k = 0; k < n_pass; ++k) keep = keep && pass_keeps(p.crop.pass[k], x[i], y[i], z[i], it[i]);
      }
      if (OBOX) {
        // the first CropBox stage removes non-finite points when its input is not dense: with no pass in front, that is
        // the segment's own flag (PCL marks every filter output dense)
        if (n_pass == 0 && !dense) keep = keep && fin;
        if (__any_sync(0xFFFFFFFFu, keep))
          for (uint32_t k = 0; k < n_obox; ++k) keep = keep & obox_keeps(sbox[k], x[i], y[i], z[i]);
      }
      fold = keep && fin;
      inv_run += __popc(__ballot_sync(0xFFFFFFFFu, keep && !fin));
    }
    minmax_if(fold, x[i], mn0, mx0);
    minmax_if(fold, y[i], mn1, mx1);
    minmax_if(fold, z[i], mn2, mx2);
    ballots[i] = __ballot_sync(0xFFFFFFFFu, keep);
    keep_bits |= (keep ? 1u : 0u) << i;
  }
  uint32_t warp_run = 0;
#pragma unroll
  for (int i = 0; i < IPT; ++i) warp_run += __popc(ballots[i]);

  // ---- bounding box of the survivors (pcl::getMinMax3D): one integer max-reduction per bound on the order-preserving
  // encodings (REDUX) instead of five shuffle rounds on six floats
  const uint32_t e0 = __reduce_max_sync(0xFFFFFFFFu, ~f32_order_enc(__float_as_uint(mn0)));
  const uint32_t e1 = __reduce_max_sync(0xFFFFFFFFu, ~f32_order_enc(__float_as_uint(mn1)));
  const uint32_t e2 = __reduce_max_sync(0xFFFFFFFFu, ~f32_order_enc(__float_as_uint(mn2)));
  const uint32_t e3 = __reduce_max_sync(0xFFFFFFFFu, f32_order_enc(__float_as_uint(mx0)));
  const uint32_t e4 = __reduce_max_sync(0xFFFFFFFFu, f32_order_enc(__float_as_uint(mx1)));
  const uint32_t e5 = __reduce_max_sync(0xFFFFFFFFu, f32_order_enc(__float_as_uint(mx2)));
  if (lane == 0) {
    s_warp_tot[warp] = warp_run;
    s_warp_inv[warp] = inv_run;
    s_mm[warp][0] = e0; s_mm[warp][1] = e1; s_mm[warp][2] = e2;
    s_mm[warp][3] = e3; s_mm[warp][4] = e4; s_mm[warp][5] = e5;
  }
  K1_TRACE(1);
  __syncthreads();
  K1_TRACE(2);

  // ---- tile-local compaction: positions inside the tile's own slot range; the dense offset comes from k_tile_scan -----
  // every warp scans the (<= 32) warp totals with shuffles: lane w holds warp w's count
  uint32_t tot, inv, pos;
  {
    const uint32_t c = lane < (uint32_t)WARPS ? s_warp_tot[lane] : 0u;
    const uint32_t incl = warp_incl_scan_u32(c);
    pos = __shfl_sync(0xFFFFFFFFu, incl - c, warp);
    tot = __shfl_sync(0xFFFFFFFFu, incl, 31);
    inv = 0;
    if (!BOX) inv = warp_sum_u32(lane < (uint32_t)WARPS ? s_warp_inv[lane] : 0u);
  }
  const uint32_t slot0 = sg->slot_base + pt0;
  if (warp == 0) {
    const uint32_t frame = sg->frame;
    if (lane == 0) {
      TileRec rec;
      rec.count = tot; rec.slot0 = slot0; rec.frame = frame; rec.dense0 = 0;
      *reinterpret_cast<uint4*>(p.tile_rec + tile) = *reinterpret_cast<const uint4*>(&rec);
      if (inv) {
        atomicAdd(&p.acc[frame].n_invalid, inv);
        atomicOr(&p.ctrl->has_invalid, 1u);
      }
    }
    if (tot > inv && lane < 6) {  // at least one finite survivor: fold the tile's box into the frame's (lane k: bound k)
      uint32_t e = s_mm[0][lane];
#pragma unroll
      for (int w = 1; w < WARPS; ++w) e = max(e, s_mm[w][lane]);
      FrameAcc* fa = p.acc + frame;
      atomicMax(lane < 3 ? &fa->nmin_enc[lane] : &fa->max_enc[lane - 3], e);
    }
  }
  K1_TRACE(3);

  // ---- write the survivors, in input order, at the head of the tile's slot range -----------------------------------------
  pos += slot0;
  const uint32_t src0 = sg->src_base + pt0 + li0;
  const uint32_t lt = lanemask_lt();
  const bool want_src = p.surv_src != nullptr;
  const uint32_t fbits = KEYS ? (sg->frame << p.box.idx_bits) : 0u;
#pragma unroll
  for (int i = 0; i < IPT; ++i) {
    if (keep_bits & (1u << i)) {
      const uint32_t q = pos + __popc(ballots[i] & lt);
      p.surv_xyzi[q] = make_float4(x[i], y[i], z[i], it[i]);
      if (want_src) p.surv_src[q] = src0 + 32 * i;
      if (KEYS) {
        // PCL: ijk = floor(p * inv_leaf) - min_b with a separately rounded multiply; here against the box grid's origin
        const uint32_t i0 = (uint32_t)(__float2int_rd(__fmul_rn(x[i], p.box.inv[0])) - p.box.min_b[0]);
        const uint32_t i1 = (uint32_t)(__float2int_rd(__fmul_rn(y[i], p.box.inv[1])) - p.box.min_b[1]);
        const uint32_t i2 = (uint32_t)(__float2int_rd(__fmul_rn(z[i], p.box.inv[2])) - p.box.min_b[2]);
        const uint32_t key = fbits | (i0 + i1 * p.box.mul1 + i2 * p.box.mul2);
        p.surv_key[q] = key;
        atomicAdd(&s_hist[key & (CM_RADIX - 1)], 1u);
      }
    }
    pos += __popc(ballots[i]);
  }
  if (KEYS) {  // this tile's digit counts -> the run's (or, frame by frame, the frame's) pass-0 histogram (fire-and-forget
               // reductions; empty bins cost nothing)
    __syncthreads();
    if (tid < CM_RADIX) {
      const uint32_t c = s_hist[tid];
      if (c) atomicAdd(p.hist + sg->frame * p.hist_frame_stride + tid, c);
    }
  }
  K1_TRACE(5);
}

template <int THREADS, int IPT, bool OBOX>
cudaError_t launch_cfg(const K1Params& p, int mode, int box, uint32_t smem, cudaStream_t stream) {
  const bool keys = p.surv_key != nullptr && box != 0;
#define CM_K1_LAUNCH(MODE, BOX, KEYS) k_transform_crop<THREADS, IPT, MODE, BOX, KEYS, OBOX><<<p.n_tiles, THREADS, smem, stream>>>(p)
#define CM_K1_BOX(MODE) do { if (box == 1) { if (keys) CM_K1_LAUNCH(MODE, 1, true); else CM_K1_LAUNCH(MODE, 1, false); } \
                             else if (box == 2) { if (keys) CM_K1_LAUNCH(MODE, 2, true); else CM_K1_LAUNCH(MODE, 2, false); } \
                             else CM_K1_LAUNCH(MODE, 0, false); } while (0)
  if (mode == (int)SEG_PACKED16) CM_K1_BOX((int)SEG_PACKED16);
  else if (mode == (int)SEG_PCL32) CM_K1_BOX((int)SEG_PCL32);
  else CM_K1_BOX(MODE_GENERIC);
#undef CM_K1_BOX
#undef CM_K1_LAUNCH
  return cudaGetLastError();
}

}  // namespace

// Two tile shapes: large batches use 4096-point tiles (fewer, fatter links in the look-back chain), single frames use
// 1024-point tiles so that a 128k-point cloud still spreads over the whole chip.
uint32_t k1_tile_points(int64_t total_points) {
  static const int forced = getenv("CM_K1_TILE") ? atoi(getenv("CM_K1_TILE")) : 0;  // debug override
  if (forced == 1024 || forced == 4096) return (uint32_t)forced;
  return total_points >= (int64_t)K1_BIG_BATCH_POINTS ? 4096u : 1024u;
}
uint32_t k1_min_tile_points() { return 1024u; }
uint32_t k1_staged_smem(uint32_t tile_points, uint32_t max_step) { return tile_points * max_step + 16u; }

cudaError_t configure_device_kernels() {
  const int big = 200 * 1024;  // the host falls back to 1024-point tiles when a staged layout needs more
  const int small = (int)k1_staged_smem(1024u, CM_MAX_STAGED_STEP);
  cudaError_t e;
#define CM_K1_ATTR(T, I, B, K, BYTES)                                                                                            \
  e = cudaFuncSetAttribute(k_transform_crop<T, I, MODE_GENERIC, B, K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, BYTES); \
  if (e != cudaSuccess) return e;                                                                                                  \
  e = cudaFuncSetAttribute(k_transform_crop<T, I, MODE_GENERIC, B, K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, BYTES);  \
  if (e != cudaSuccess) return e;
  CM_K1_ATTR(512, 8, 0, false, big) CM_K1_ATTR(512, 8, 1, false, big) CM_K1_ATTR(512, 8, 2, false, big)
  CM_K1_ATTR(512, 8, 1, true, big) CM_K1_ATTR(512, 8, 2, true, big)
  CM_K1_ATTR(256, 4, 0, false, small) CM_K1_ATTR(256, 4, 1, false, small) CM_K1_ATTR(256, 4, 2, false, small)
  CM_K1_ATTR(256, 4, 1, true, small) CM_K1_ATTR(256, 4, 2, true, small)
#undef CM_K1_ATTR
  return cudaSuccess;
}

cudaError_t launch_transform_crop(const K1Params& p, uint32_t tile_points, int mode, uint32_t staged_smem_bytes,
                                  cudaStream_t stream) {
  if (p.n_tiles == 0) return cudaSuccess;
  const int box = p.crop.is_box ? (p.crop.use_i ? 2 : 1) : 0;
  if (p.n_obox) {
    if (tile_points == 4096u) return launch_cfg<512, 8, true>(p, mode, box, staged_smem_bytes, stream);
    return launch_cfg<256, 4, true>(p, mode, box, staged_smem_bytes, stream);
  }
  if (tile_points == 4096u) return launch_cfg<512, 8, false>(p, mode, box, staged_smem_bytes, stream);
  return launch_cfg<256, 4, false>(p, mode, box, staged_smem_bytes, stream);
}

}  // namespace cm
