// cm_voxel.cu -- VoxelGrid front end (bounding box -> grid -> 64-bit voxel keys + digit histograms) and back end
// (run detection on the sorted keys -> centroid per voxel -> min-points filter -> stable compaction) for sm_100a.
//
// Replaces pcl::VoxelGrid<pcl::PointXYZI>::applyFilter as configured by the reference's voxelgrid()
// (pc_preprocessing_main.cpp:168-177, CloudFusionNode.h:276-289, PreprocessingNode.h:236-249):
//   first pass  (idx per point)             -> k_voxel_key_hist   (key = (frame << idx_bits) | idx, idx = i + j*div_x + k*div_x*div_y;
//                                              frame-segmented runs: the bare idx, the frame is the position's -- k_grid_setup
//                                              plans that, k_seg_base prepares the per-frame first positions)
//   second pass (std::sort)                 -> cm_radix_sort.cu   (onesweep LSD radix sort of key / point-index pairs)
//   third+fourth pass (runs, CentroidPoint) -> k_voxel_centroid
// The voxel index arithmetic repeats PCL's float32 formulas exactly (floorf(x * inv_leaf) with a separately rounded
// multiply); the linearisation is carried in 64 bits so clouds beyond PCL's INT32 cell limit still work.
//
// Roofline: HBM for every kernel here. Algorithmic bytes: key_hist reads 16 B and writes key_bytes per point;
// centroid reads key_bytes + 4 per point, gathers 16 B per point and writes 16/32 + 4 + 8 B per voxel.
#include "cm_kernels.h"

namespace cm {

namespace {

constexpr int VX_THREADS = 256;
constexpr int KH_IPT = 8;
constexpr int KH_TILE = VX_THREADS * KH_IPT;  // 2048 points per min/max tile
constexpr int KH_DENSE_TILE = 4096;           // virtual tile of the key kernel when the input is a plain dense cloud
constexpr int SCAN_THREADS = 1024;
#ifndef KH_UNROLL
#define KH_UNROLL 8
#endif
#ifndef CE_ASYNC_GATHER
#define CE_ASYNC_GATHER 1  // the count sweep of the next tile gathers its points by cp.async into a second buffer (0: the
#endif                     // tile's item phase reads its records again and gathers synchronously -- the round-2 kernel)
#ifndef CE_MIN_CTAS
#define CE_MIN_CTAS (CE_ASYNC_GATHER ? 3 : 4)  // two 32 KB point buffers: 70 KB per CTA, 3 CTAs per SM
#endif
#ifndef CE_PREFETCH
#define CE_PREFETCH 0   // tried: L2 prefetch of the next tile's points from the count sweep. cfg3 batch: no change (0.148 vs 0.146 ms);
#endif                  // cfg5 sweep: 17 % SLOWER (every point is gathered there and the prefetch only adds requests). Off.
                        // (CE_ASYNC_GATHER 0 only: the asynchronous gather replaces it)
#ifndef CE_LB_POLL_ONE
#define CE_LB_POLL_ONE 0
#endif
#ifndef CE_LB_POLL_NS
#define CE_LB_POLL_NS 30
#endif
constexpr int CE_IPT = 8;
constexpr int CE_TILE = VX_THREADS * CE_IPT;  // 2048 sorted items per centroid tile
constexpr int CE_PT_BUFS = CE_ASYNC_GATHER ? 2 : 1;
constexpr size_t CE_DYN_SMEM = (size_t)CE_PT_BUFS * CE_TILE * sizeof(float4);  // the point buffers (dynamic shared memory)

// 16-byte global -> shared copy that completes asynchronously (LDGSTS; .cg: cached in L2 only), and its group fences
__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(PENDING) : "memory"); }

// Exclusive scan of one value per thread over a 1024-thread block. Returns the exclusive prefix; *total = block sum.
__device__ __forceinline__ uint32_t block_excl_scan_1024(uint32_t v, uint32_t* scratch /* 33 words */, uint32_t* total) {
  const uint32_t tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
  const uint32_t incl = warp_incl_scan_u32(v);
  if (lane == 31) scratch[w] = incl;
  __syncthreads();
  if (w == 0) {
    const uint32_t t = scratch[lane];
    const uint32_t ti = warp_incl_scan_u32(t);
    scratch[lane] = ti - t;
    if (lane == 31) scratch[32] = ti;
  }
  __syncthreads();
  const uint32_t res = incl - v + scratch[w];
  *total = scratch[32];
  __syncthreads();
  return res;
}

}  // namespace

// ---- pcl::getMinMax3D on a plain packed cloud (VoxelGrid-only entry) -------------------------------------------------
__global__ void __launch_bounds__(VX_THREADS) k_minmax(const float4* __restrict__ pts, uint32_t n, Ctrl* ctrl,
                                                       FrameAcc* acc, uint32_t* frame_surv_start) {
  __shared__ float s_mm[VX_THREADS / 32][6];
  __shared__ uint32_t s_inv[VX_THREADS / 32];
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  float mn0 = 3.402823466e+38f, mn1 = mn0, mn2 = mn0, mx0 = -mn0, mx1 = -mn0, mx2 = -mn0;
  uint32_t inv = 0, fin_cnt = 0;
  for (size_t i = (size_t)blockIdx.x * VX_THREADS + tid; i < n; i += (size_t)gridDim.x * VX_THREADS) {
    const float4 v = ldg_stream_f4(pts + i);
    if (finite_f32(v.x) && finite_f32(v.y) && finite_f32(v.z)) {
      mn0 = fminf(mn0, v.x); mx0 = fmaxf(mx0, v.x);
      mn1 = fminf(mn1, v.y); mx1 = fmaxf(mx1, v.y);
      mn2 = fminf(mn2, v.z); mx2 = fmaxf(mx2, v.z);
      ++fin_cnt;
    } else {
      ++inv;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn0 = fminf(mn0, __shfl_xor_sync(0xFFFFFFFFu, mn0, o)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xFFFFFFFFu, mx0, o));
    mn1 = fminf(mn1, __shfl_xor_sync(0xFFFFFFFFu, mn1, o)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xFFFFFFFFu, mx1, o));
    mn2 = fminf(mn2, __shfl_xor_sync(0xFFFFFFFFu, mn2, o)); mx2 = fmaxf(mx2, __shfl_xor_sync(0xFFFFFFFFu, mx2, o));
  }
  inv = warp_sum_u32(inv);
  fin_cnt = warp_sum_u32(fin_cnt);
  if (lane == 0) {
    s_mm[warp][0] = mn0; s_mm[warp][1] = mn1; s_mm[warp][2] = mn2;
    s_mm[warp][3] = mx0; s_mm[warp][4] = mx1; s_mm[warp][5] = mx2;
    s_inv[warp] = inv;
    if (fin_cnt == 0) s_mm[warp][0] = 3.402823466e+38f;  // keeps the fold below neutral
  }
  __syncthreads();
  if (tid == 0) {
    float a0 = s_mm[0][0], a1 = s_mm[0][1], a2 = s_mm[0][2], b0 = s_mm[0][3], b1 = s_mm[0][4], b2 = s_mm[0][5];
    uint32_t ti = s_inv[0];
    for (int w = 1; w < VX_THREADS / 32; ++w) {
      a0 = fminf(a0, s_mm[w][0]); a1 = fminf(a1, s_mm[w][1]); a2 = fminf(a2, s_mm[w][2]);
      b0 = fmaxf(b0, s_mm[w][3]); b1 = fmaxf(b1, s_mm[w][4]); b2 = fmaxf(b2, s_mm[w][5]);
      ti += s_inv[w];
    }
    if (b0 >= a0) {  // at least one finite point seen by this block
      atomicMax(&acc->nmin_enc[0], ~f32_order_enc(__float_as_uint(a0)));
      atomicMax(&acc->nmin_enc[1], ~f32_order_enc(__float_as_uint(a1)));
      atomicMax(&acc->nmin_enc[2], ~f32_order_enc(__float_as_uint(a2)));
      atomicMax(&acc->max_enc[0], f32_order_enc(__float_as_uint(b0)));
      atomicMax(&acc->max_enc[1], f32_order_enc(__float_as_uint(b1)));
      atomicMax(&acc->max_enc[2], f32_order_enc(__float_as_uint(b2)));
    }
    if (ti) {
      atomicAdd(&acc->n_invalid, ti);
      atomicOr(&ctrl->has_invalid, 1u);
    }
    if (blockIdx.x == 0) {
      frame_surv_start[0] = 0;
      frame_surv_start[1] = n;
    }
  }
}

// ---- one CTA: dense offsets of the K1 tiles, frame / segment starts, total ------------------------------------------------
__device__ __forceinline__ void tile_scan_body(TileRec* __restrict__ rec, uint32_t n_tiles, const SegDev* __restrict__ segs,
                                               uint32_t n_seg, uint32_t n_frames, uint32_t* frame_surv_start,
                                               uint32_t* seg_surv_start, uint32_t* s_scr /* 33 words */) {
  const uint32_t tid = threadIdx.x;
  const uint32_t chunk = (n_tiles + SCAN_THREADS - 1) / SCAN_THREADS;
  const uint32_t b = min(n_tiles, tid * chunk), e = min(n_tiles, b + chunk);
  // a single CTA is latency-bound: the counts of a thread's chunk are fetched eight at a time (independent loads) and,
  // for chunks of up to eight tiles (batches of up to 8192 tiles), kept in registers for the second sweep
  constexpr int W = 8;
  uint32_t c[W];
  uint32_t sum = 0;
  for (uint32_t i0 = b; i0 < e; i0 += W) {
#pragma unroll
    for (int k = 0; k < W; ++k) c[k] = (i0 + k < e) ? rec[i0 + k].count : 0u;
#pragma unroll
    for (int k = 0; k < W; ++k) sum += c[k];
  }
  uint32_t total;
  uint32_t run = block_excl_scan_1024(sum, s_scr, &total);
  if (chunk <= (uint32_t)W) {
#pragma unroll
    for (int k = 0; k < W; ++k) {
      if (b + k < e) rec[b + k].dense0 = run;
      run += c[k];
    }
  } else {
    for (uint32_t i = b; i < e; ++i) {
      const uint32_t cc = rec[i].count;
      rec[i].dense0 = run;
      run += cc;
    }
  }
  __syncthreads();  // dense0 of every tile is visible to the block
  for (uint32_t s = tid; s < n_seg; s += SCAN_THREADS) {
    const uint32_t d0 = rec[segs[s].tile_begin].dense0;
    seg_surv_start[s] = d0;
    if (segs[s].first_of_frame) frame_surv_start[segs[s].frame] = d0;
  }
  if (tid == 0) frame_surv_start[n_frames] = total;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_tile_scan(TileRec* __restrict__ rec, uint32_t n_tiles,
                                                           const SegDev* __restrict__ segs, uint32_t n_seg,
                                                           uint32_t n_frames, uint32_t* frame_surv_start,
                                                           uint32_t* seg_surv_start) {
  __shared__ uint32_t s_scr[33];
  tile_scan_body(rec, n_tiles, segs, n_seg, n_frames, frame_surv_start, seg_surv_start, s_scr);
}

// ---- dense copy of the merged cropped cloud, on request ---------------------------------------------------------------------
__global__ void __launch_bounds__(VX_THREADS) k_compact_survivors(const TileRec* __restrict__ rec, uint32_t n_tiles,
                                                                 const float4* __restrict__ slot_xyzi,
                                                                 const uint32_t* __restrict__ slot_src,
                                                                 float4* __restrict__ dense_xyzi,
                                                                 uint32_t* __restrict__ dense_src,
                                                                 uint32_t* __restrict__ dense_slot) {
  for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const TileRec r = rec[t];
    for (uint32_t j = threadIdx.x; j < r.count; j += VX_THREADS) {
      dense_xyzi[r.dense0 + j] = slot_xyzi[r.slot0 + j];
      if (dense_src) dense_src[r.dense0 + j] = slot_src[r.slot0 + j];
      if (dense_slot) dense_slot[r.dense0 + j] = r.slot0 + j;
    }
  }
}

// ---- fold externally supplied bounds (the all-reduced bounding box of a cloud partitioned over several GPUs) into frame 0 --
__global__ void k_seed_bounds(FrameAcc* acc, float mn0, float mn1, float mn2, float mx0, float mx1, float mx2) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    atomicMax(&acc->nmin_enc[0], ~f32_order_enc(__float_as_uint(mn0)));
    atomicMax(&acc->nmin_enc[1], ~f32_order_enc(__float_as_uint(mn1)));
    atomicMax(&acc->nmin_enc[2], ~f32_order_enc(__float_as_uint(mn2)));
    atomicMax(&acc->max_enc[0], f32_order_enc(__float_as_uint(mx0)));
    atomicMax(&acc->max_enc[1], f32_order_enc(__float_as_uint(mx1)));
    atomicMax(&acc->max_enc[2], f32_order_enc(__float_as_uint(mx2)));
  }
}

// ---- grid per frame + sort plan (one block) -----------------------------------------------------------------------
// PCL 1.8.1: min_b = floor(min_p * inv), max_b = floor(max_p * inv), div_b = max_b - min_b + 1, and the guard
// dx*dy*dz > INT32_MAX with d = (int64)((max_p - min_p) * inv) + 1.
// When the survivors come out of K1 the same CTA first turns the K1 tile counts into dense offsets (tile_scan_body):
// one launch and one dependent-launch gap less on the critical path.
struct TileScanArgs {
  TileRec* rec;
  uint32_t n_tiles;
  const SegDev* segs;
  uint32_t n_seg;
  uint32_t* seg_surv_start;
};
__global__ void __launch_bounds__(SCAN_THREADS) k_grid_setup(const VoxelParams p, const TileScanArgs ts) {
  __shared__ uint32_t s_maxbits;
  __shared__ uint32_t s_scr[33];
  const uint32_t tid = threadIdx.x;
  if (tid == 0) s_maxbits = 0;
  if (ts.rec) tile_scan_body(ts.rec, ts.n_tiles, ts.segs, ts.n_seg, p.n_frames, const_cast<uint32_t*>(p.frame_surv_start),
                             ts.seg_surv_start, s_scr);
  __syncthreads();
  if (ts.rec && p.fused_keys && !p.box.seg_sort) {
    // which K1 tile holds the first key of every radix tile (pass 0 reads the keys where K1 left them): a K1 tile has at
    // most 4096 survivors, fewer than a radix tile, so at most one radix-tile boundary falls into it
    const unsigned long long T = p.sort_tile;
    for (uint32_t i = tid; i < ts.n_tiles; i += SCAN_THREADS) {
      const uint32_t c = ts.rec[i].count;
      if (!c) continue;
      const unsigned long long d0 = ts.rec[i].dense0;
      const unsigned long long t = (d0 + T - 1ull) / T;
      if (t * T < d0 + c) p.first_k1[t] = i;
    }
  }
  for (uint32_t f = tid; f < p.n_frames; f += SCAN_THREADS) {
    const FrameAcc a = p.acc[f];
    GridDev g;
    g.pcl_overflow = 0;
    g.bits = 0;
    g.mul1 = 0;
    g.mul2 = 0;
    g.zero_keys = 0;
    g.empty = (a.max_enc[0] == 0u && a.nmin_enc[0] == 0u) ? 1u : 0u;
    if (g.empty) {
      for (int k = 0; k < 3; ++k) { g.min_b[k] = 0; g.max_b[k] = 0; g.div_b[k] = 0; }
    } else {
      long long d[3];
      unsigned long long div[3];
      bool range_err = false;
      for (int k = 0; k < 3; ++k) {
        const float mn = __uint_as_float(f32_order_dec(~a.nmin_enc[k]));
        const float mx = __uint_as_float(f32_order_dec(a.max_enc[k]));
        const float inv = p.inv_leaf[k];
        d[k] = __float2ll_rz(__fmul_rn(__fsub_rn(mx, mn), inv)) + 1ll;
        const float fmn = floorf(__fmul_rn(mn, inv)), fmx = floorf(__fmul_rn(mx, inv));
        // coordinates are limited to +-2^30 cells so that the int32 grid origin is exact
        if (!(fabsf(fmn) < 1073741824.f) || !(fabsf(fmx) < 1073741824.f)) range_err = true;
        g.min_b[k] = (int)fmn;
        g.max_b[k] = (int)fmx;
        const long long dv = (long long)g.max_b[k] - (long long)g.min_b[k] + 1ll;
        g.div_b[k] = (int)dv;
        div[k] = (unsigned long long)dv;
        if (dv > (1ll << 21)) range_err = true;
      }
      const long long imax = 2147483647ll;
      bool ovf = d[0] > imax || d[1] > imax || d[2] > imax || d[0] < 0 || d[1] < 0 || d[2] < 0;
      if (!ovf) {
        const long long p01 = d[0] * d[1];
        ovf = p01 > imax || p01 * d[2] > imax;
      }
      g.pcl_overflow = ovf ? 1 : 0;
      if (range_err) {
        // No key of such a frame can be formed, so every point gets index 0 of a 1-cell grid: keys stay below the frame's
        // limit whatever idx_bits comes out (0 when no frame has a usable grid), and no kernel derives a frame from garbage.
        // Overflow mode 1 returns a frame PCL refuses as its cropped cloud: its voxels are not used, so no error then.
        if (!(p.pcl_refuses && ovf)) atomicExch(&p.ctrl->error, (uint32_t)CM_DEV_E_KEY_RANGE);
        div[0] = div[1] = div[2] = 1;
        g.zero_keys = 1;
      }
      g.mul1 = div[0];
      g.mul2 = div[0] * div[1];
      const unsigned long long cells = div[0] * div[1] * div[2];
      g.bits = cells <= 1ull ? 0u : (uint32_t)(64 - __clzll((long long)(cells - 1ull)));
      atomicMax(&s_maxbits, g.bits);
    }
    p.grid[f] = g;
  }
  __syncthreads();
  // the run epoch of the look-back words (30 bits): on wrap-around clear the words and start over
  {
    const uint32_t e = *p.epoch_dev;
    const bool wrap = e + 64u >= (1u << 30);
    if (wrap) {
      for (uint32_t i = tid; i < p.lb_sort_words; i += SCAN_THREADS) p.lb_sort[i] = 0ull;
      for (uint32_t i = tid; i < p.cent_status_words; i += SCAN_THREADS) p.cent_status[i] = 0ull;
    }
    __syncthreads();
    if (tid == 0) *p.epoch_dev = wrap ? 16u : e + 16u;
  }
  __shared__ SortInfo s_si;
  if (tid == 0) {
    const bool has_invalid = p.ctrl->has_invalid != 0u;
    const uint32_t key_frames = p.n_frames + (has_invalid ? 1u : 0u);
    uint32_t frame_bits = key_frames <= 1u ? 0u : (uint32_t)(32 - __clz((int)(key_frames - 1u)));
    uint32_t idx_bits = s_maxbits;
    if (p.fused_keys) idx_bits = p.box.idx_bits;  // the keys K1 wrote are built on the crop box's grid, which holds every frame's
    // Frame-segmented sort: the batch is frame-ordered, so the frame bits need no sorting. Possible when no survivor is
    // non-finite (those are keyed into a sentinel frame of their own) and the voxel index alone fits 32 bits -- which PCL
    // itself requires of a frame it filters.
    bool seg = p.segmented == 2u;
    if (p.segmented == 1u) seg = !has_invalid && idx_bits <= 32u;
    if (seg) frame_bits = 0u;
    // a fused-key run planned frame by frame (BoxGrid::seg_sort) keeps its frame bits in the keys but ranks none of them
    const bool fused_seg = p.fused_keys && p.box.seg_sort;
    uint32_t width = p.key_bytes;
    if (p.dual_width) width = p.segmented == 1u ? (seg ? 4u : 8u) : (frame_bits + idx_bits <= 32u ? 4u : 8u);
    uint32_t total = frame_bits + idx_bits;
    if (total > width * 8u) {
      atomicExch(&p.ctrl->error, (uint32_t)CM_DEV_E_KEY_RANGE);
      total = width * 8u;
      idx_bits = total - frame_bits;
    }
    uint32_t passes = fused_seg ? p.box.n_pass : (total + CM_RADIX_BITS - 1) / CM_RADIX_BITS;
    if (passes == 0) passes = 1;
    if (passes > p.max_passes) {  // the host enqueued fewer pass launches than the data needs
      atomicExch(&p.ctrl->error, (uint32_t)CM_DEV_E_KEY_RANGE);
      passes = p.max_passes;
    }
    SortInfo si;
    si.num_passes = passes;
    si.total_bits = total;
    si.idx_bits = idx_bits;
    si.n_keys = p.frame_surv_start[p.n_frames];
    si.key_frames = key_frames;
    si.width = width;
    si.segmented = seg ? 1u : 0u;
    si.n_seg_tiles = 0;
    si.seg_sort = (seg || fused_seg) ? 1u : 0u;
    s_si = si;
  }
  __syncthreads();
  if (s_si.seg_sort) {
    // the frame-aligned radix tiles: frame f owns ceil(n_f / T) consecutive tiles
    const uint32_t T = p.sort_tile, F = p.n_frames;
    uint32_t carry = 0;
    for (uint32_t f0 = 0; f0 < F; f0 += SCAN_THREADS) {
      const uint32_t f = f0 + tid;
      const uint32_t nf = f < F ? p.frame_surv_start[f + 1] - p.frame_surv_start[f] : 0u;
      uint32_t tot;
      const uint32_t ex = block_excl_scan_1024((nf + T - 1u) / T, s_scr, &tot);
      if (f < F) p.seg_frame_tile0[f] = carry + ex;
      carry += tot;
    }
    if (tid == 0) { p.seg_frame_tile0[F] = carry; s_si.n_seg_tiles = carry; }
    __syncthreads();
    const uint32_t warp = tid >> 5, lane = tid & 31u;
    for (uint32_t f = warp; f < F; f += SCAN_THREADS / 32) {
      const uint32_t b = p.frame_surv_start[f], e = p.frame_surv_start[f + 1];
      const uint32_t t0 = p.seg_frame_tile0[f], nt = p.seg_frame_tile0[f + 1] - t0;
      for (uint32_t t = lane; t < nt; t += 32u) {
        SegTile st;
        st.base = b + t * T;
        st.n = min(T, e - st.base);
        st.frame = f | (t == 0u ? CM_SEG_FIRST : 0u);
        st.pad = 0u;
        p.seg_tile[t0 + t] = st;
      }
    }
    if (p.fused_keys) {
      // which K1 tile holds the first key of every radix tile (a K1 tile lies in one frame and has fewer survivors than a
      // radix tile, so at most one tile start of its frame falls into it) ...
      for (uint32_t i = tid; i < ts.n_tiles; i += SCAN_THREADS) {
        const TileRec r = ts.rec[i];
        if (!r.count) continue;
        const uint32_t fs = p.frame_surv_start[r.frame];
        const uint32_t t = (r.dense0 - fs + T - 1u) / T;
        if (fs + (unsigned long long)t * T < (unsigned long long)r.dense0 + r.count) p.first_k1[p.seg_frame_tile0[r.frame] + t] = i;
      }
      // ... and the frames' first positions of pass 0 from the digit counts K1 left in seg_hist (one warp per frame)
      for (uint32_t f = warp; f < F; f += SCAN_THREADS / 32) {
        uint32_t* h = p.seg_hist + (size_t)f * (CM_SEG_PASSES * CM_RADIX) + lane * 8u;
        uint32_t c[8], sum = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) { c[k] = h[k]; sum += c[k]; }
        uint32_t run = p.frame_surv_start[f] + warp_incl_scan_u32(sum) - sum;
#pragma unroll
        for (int k = 0; k < 8; ++k) { h[k] = run; run += c[k]; }
      }
    }
    // ... and which frames every tile of the centroid pass touches (nearly always one: no search per item there)
    const uint32_t M = s_si.segmented ? s_si.n_keys : 0u;
    auto frame_from = [&](uint32_t i, uint32_t lo) {  // the last frame that starts at or before position i
      uint32_t hi = F - 1u;
      while (lo < hi) {
        const uint32_t mid = (lo + hi + 1u) >> 1;
        if (p.frame_surv_start[mid] <= i) lo = mid; else hi = mid - 1u;
      }
      return lo;
    };
    for (uint32_t t = tid; (unsigned long long)t * CE_TILE < M; t += SCAN_THREADS) {
      const uint32_t b = t * CE_TILE, e = min(b + (uint32_t)CE_TILE, M);
      const uint32_t lo = frame_from(b, 0u);
      p.seg_cent_range[t] = make_uint2(lo, frame_from(e - 1u, lo));
    }
    __syncthreads();
  }
  if (tid == 0) *p.info = s_si;
}

// ---- voxel key per point + the digit histograms of every radix pass -----------------------------------------------------
// Walks the K1 tiles: tile t contributes rec.count survivors read from slots [slot0, slot0+count) and written densely at
// [dense0, dense0+count): key = (frame << idx_bits) | idx, value = slot (what the centroid pass gathers by).
// Histograms: one shared-memory increment per key and pass. The hardware aggregates lanes that hit the same counter
// (SASS ATOMS.POPC.INC), so neither the warp-uniform high digits nor the scattered low digits need software matching.
// CHECK: non-finite survivors are possible (no crop pass configured) and get the sentinel frame; any PassThrough stage
// rejects them, so the common instantiation carries no finite tests.
// SEG (frame-segmented sort): the key is the voxel index alone, and the digits are counted per frame -- the counters are
// flushed to the frame's own histogram whenever the CTA moves on to a tile of another frame.
template <typename KeyT, bool CHECK, bool SEG = false>
__device__ __forceinline__ void key_hist_tiles(const VoxelParams& p, uint32_t (*s_hist)[CM_RADIX], const SortInfo& si,
                                               uint32_t M) {
  const uint32_t tid = threadIdx.x;
  const uint32_t F = p.n_frames;
  const uint32_t n_pass = si.num_passes, idx_bits = si.idx_bits;
  const bool dense = p.tile_rec == nullptr;
  // dense input (no K1 tiles): frame f is the range [frame_surv_start[f], frame_surv_start[f+1]) and owns its own tiles
  uint32_t n_tiles = p.n_k1_tiles;
  if (dense) {
    n_tiles = 0;
    for (uint32_t f = 0; f < F; ++f)
      n_tiles += (p.frame_surv_start[f + 1] - p.frame_surv_start[f] + KH_DENSE_TILE - 1) / KH_DENSE_TILE;
  }
  KeyT* __restrict__ keys = reinterpret_cast<KeyT*>(p.keys_a);
  uint32_t* __restrict__ vals = p.vals_a;
  uint2* __restrict__ recs = reinterpret_cast<uint2*>(p.keys_a);
  const unsigned long long sentinel = (unsigned long long)F << idx_bits;
  const float inv0 = p.inv_leaf[0], inv1 = p.inv_leaf[1], inv2 = p.inv_leaf[2];

  uint32_t hist_frame = 0xFFFFFFFFu;  // SEG: the frame the shared counters belong to
  auto flush_frame = [&]() {
    __syncthreads();
    if (hist_frame != 0xFFFFFFFFu) {
      uint32_t* dst = p.seg_hist + (size_t)hist_frame * (CM_SEG_PASSES * CM_RADIX);
      for (uint32_t i = tid; i < n_pass * CM_RADIX; i += VX_THREADS) {
        const uint32_t c = (&s_hist[0][0])[i];
        if (c) { atomicAdd(dst + i, c); (&s_hist[0][0])[i] = 0u; }
      }
    }
    __syncthreads();
  };
  for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    TileRec r;
    if (dense) {
      uint32_t t = tile, f = 0, f_begin = 0, f_end = 0;
      for (; f < F; ++f) {
        f_begin = p.frame_surv_start[f]; f_end = p.frame_surv_start[f + 1];
        const uint32_t tf = (f_end - f_begin + KH_DENSE_TILE - 1) / KH_DENSE_TILE;
        if (t < tf) break;
        t -= tf;
      }
      r.frame = f; r.slot0 = f_begin + t * KH_DENSE_TILE; r.dense0 = r.slot0;
      r.count = min((uint32_t)KH_DENSE_TILE, f_end - r.slot0);
    } else {
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(p.tile_rec + tile));
      r.count = q.x; r.slot0 = q.y; r.frame = q.z; r.dense0 = q.w;
    }
    if (r.count == 0) continue;
    if (SEG && r.frame != hist_frame) {
      flush_frame();
      hist_frame = r.frame;
    }
    const GridDev* __restrict__ g = p.grid + r.frame;
    const KeyT fbits = SEG ? (KeyT)0 : (KeyT)((unsigned long long)r.frame << idx_bits);
    const KeyT mul1 = (KeyT)g->mul1, mul2 = (KeyT)g->mul2;  // 32-bit arithmetic when the key is 32-bit
    const KeyT idx_keep = g->zero_keys ? (KeyT)0 : ~(KeyT)0;  // a frame without a usable grid: index 0 (see k_grid_setup)
    const int mb0 = g->min_b[0], mb1 = g->min_b[1], mb2 = g->min_b[2];
    const float4* __restrict__ src = p.pts + r.slot0;
    constexpr int U = KH_UNROLL;  // points per thread in flight
    for (uint32_t j0 = 0; j0 < r.count; j0 += U * VX_THREADS) {
      const bool whole = j0 + U * VX_THREADS <= r.count;
      float4 pv[U];
      if (whole) {
#pragma unroll
        for (int u = 0; u < U; ++u) pv[u] = ldg_stream_f4(src + j0 + u * VX_THREADS + tid);
      } else {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint32_t j = j0 + u * VX_THREADS + tid;
          pv[u] = (j < r.count) ? ldg_stream_f4(src + j) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const uint32_t j = j0 + u * VX_THREADS + tid;
        if (!whole && j >= r.count) continue;
        const float4 v = pv[u];
        // PCL: ijk = (int)(floor(x * inv) - (float)min_b); here in integers (identical below 2^24 cells)
        const KeyT i0 = (KeyT)(__float2int_rd(__fmul_rn(v.x, inv0)) - mb0);
        const KeyT i1 = (KeyT)(__float2int_rd(__fmul_rn(v.y, inv1)) - mb1);
        const KeyT i2 = (KeyT)(__float2int_rd(__fmul_rn(v.z, inv2)) - mb2);
        KeyT key = fbits | ((KeyT)(i0 + i1 * mul1 + i2 * mul2) & idx_keep);
        if (CHECK && !(finite_f32(v.x) && finite_f32(v.y) && finite_f32(v.z))) key = (KeyT)sentinel;
        if (sizeof(KeyT) == 4) {  // 32-bit keys travel as 8-byte (key, value) records
          recs[r.dense0 + j] = make_uint2((uint32_t)key, r.slot0 + j);
        } else {
          keys[r.dense0 + j] = key;
          vals[r.dense0 + j] = r.slot0 + j;
        }
        if (sizeof(KeyT) == 4) {
#pragma unroll
          for (uint32_t ps = 0; ps < 4; ++ps)
            if (ps < n_pass) atomicAdd(&s_hist[ps][((uint32_t)key >> (ps * CM_RADIX_BITS)) & (CM_RADIX - 1)], 1u);
        } else {
#pragma unroll
          for (uint32_t ps = 0; ps < CM_MAX_SORT_PASSES; ++ps)
            if (ps < n_pass)
              atomicAdd(&s_hist[ps][(uint32_t)((unsigned long long)key >> (ps * CM_RADIX_BITS)) & (CM_RADIX - 1)], 1u);
        }
      }
    }
  }
  if (SEG) flush_frame();
}

template <typename KeyT>
__global__ void __launch_bounds__(VX_THREADS) k_voxel_key_hist(const VoxelParams p) {
  __shared__ uint32_t s_hist[CM_MAX_SORT_PASSES][CM_RADIX];
  const uint32_t tid = threadIdx.x;
  const SortInfo si = *p.info;
  if (p.dual_width && ((si.width == 4u) != (sizeof(KeyT) == 4))) return;  // the other key width runs
  for (uint32_t i = tid; i < CM_MAX_SORT_PASSES * CM_RADIX; i += VX_THREADS) (&s_hist[0][0])[i] = 0;
  __syncthreads();
  const uint32_t M = p.frame_surv_start[p.n_frames];
  if (sizeof(KeyT) == 4 && si.segmented) {
    key_hist_tiles<uint32_t, false, true>(p, s_hist, si, M);  // the frames' own histograms are complete: nothing global
    return;
  }
  if (si.key_frames > p.n_frames) key_hist_tiles<KeyT, true>(p, s_hist, si, M);
  else key_hist_tiles<KeyT, false>(p, s_hist, si, M);
  __syncthreads();
  for (uint32_t i = tid; i < si.num_passes * CM_RADIX; i += VX_THREADS) {
    const uint32_t c = (&s_hist[0][0])[i];
    if (c) atomicAdd(p.hist + i, c);
  }
}

// ---- segmented runs: per-frame digit counts -> where the frame's keys of digit d start in the output of pass ps ------------
// NB = CM_WIDE_BINS: a fused-key run sorted frame by frame -- passes 1.. only (k_grid_setup did pass 0), the last one of
// box.top_bins digits.
template <int NB>
__global__ void __launch_bounds__(NB) k_seg_base(const VoxelParams p) {
  __shared__ uint32_t s_scan[NB / 32 + 4];
  const SortInfo si = *p.info;
  constexpr uint32_t first_pass = NB > CM_RADIX ? 1u : 0u;
  if (!si.seg_sort || blockIdx.y < first_pass || blockIdx.y >= si.num_passes) return;
  const uint32_t f = blockIdx.x, tid = threadIdx.x;
  uint32_t* h = p.seg_hist + ((size_t)f * CM_SEG_PASSES + blockIdx.y) * CM_RADIX;
  const uint32_t nb = (NB > CM_RADIX && blockIdx.y + 1u == si.num_passes) ? p.box.top_bins : CM_RADIX;
  uint32_t tot;
  const uint32_t ex = block_excl_scan<NB>(tid < nb ? h[tid] : 0u, s_scan, &tot);
  if (tid < nb) h[tid] = p.frame_surv_start[f] + ex;
}

// segmented runs sort (idx, slot) records; callers of cm_get_device_out get (frame << idx_bits | idx) and the slots
__global__ void __launch_bounds__(VX_THREADS) k_seg_keys64(const uint2* __restrict__ rec, unsigned long long* __restrict__ keys,
                                                          uint32_t* __restrict__ vals, const VoxelParams p) {
  const uint32_t F = p.n_frames, idx_bits = p.info->idx_bits;
  const uint32_t* __restrict__ fss = p.frame_surv_start;
  const uint32_t n = fss[F];
  for (uint32_t i = blockIdx.x * VX_THREADS + threadIdx.x; i < n; i += gridDim.x * VX_THREADS) {
    uint32_t lo = 0, hi = F - 1u;  // the last frame that starts at or before i
    while (lo < hi) {
      const uint32_t mid = (lo + hi + 1u) >> 1;
      if (fss[mid] <= i) lo = mid; else hi = mid - 1u;
    }
    const uint2 r = rec[i];
    keys[i] = ((unsigned long long)lo << idx_bits) | (unsigned long long)r.x;
    vals[i] = r.y;
  }
}

// ---- runs of equal key -> centroid, min-points filter, order-preserving compaction ----------------------------------
// The radix sort is stable and started from ascending point order, so inside a run the points are in ascending index
// order: the float accumulation below is sequential in that order (one valid order of PCL's CentroidPoint loop, whose
// own order is unspecified because std::sort is unstable). centroid = sum / (float)n with an IEEE division.
//
// The voxels leave the kernel dense and in order: a tile publishes its voxel count as soon as it is known and obtains the
// number of voxels of all earlier tiles by a decoupled look-back (one warp, 32 tiles per round, epoch-tagged words) that runs
// while the other warps already sum their first voxel -- the separate scan + compaction launches (and the 56 bytes per voxel
// they moved) are gone. Tiles are handed out by an arrival ticket, so a tile only ever waits for tiles that are running.
//
// Two phases per 2048-item tile, both with every lane busy:
//   per item  (thread t owns items 8t .. 8t+7): records in with 16-byte loads, neighbour keys by shuffle, head-of-run
//             and min-points flags as bit masks, the points of surviving runs gathered into shared memory (asynchronous
//             copies issued one tile ahead, in the count sweep below), one head bit per item into a shared bit array;
//   per voxel (thread r owns the r-th surviving run of the tile, found through the block scan of the per-thread
//             counts): end of run from the head bit array, sequential sum over shared memory (the part of a run that
//             continues past the tile is read from global memory), division, coalesced tile-local output.
// The first version did the per-voxel work in the thread that owned the head item: with ~1 surviving head per 8 items
// the warp executed the whole epilogue (four divisions, stores, atomics) for a handful of active lanes at a time, and
// the kernel issued 190 instructions per item.
//
// SEG (frame-segmented sort): the records carry the bare voxel index; frame f occupies positions [frame_surv_start[f],
// frame_surv_start[f+1]) of the sorted array exactly as it did before the sort, so the frame of an item follows from its
// position and the kernel works on the logical key (frame << idx_bits | idx) like the unsegmented 64-bit one.
// ---- tail runs ---------------------------------------------------------------------------------------------------------------
// A run that continues past the centroid tile in which it starts is walked by the thread that owns its head, two dependent
// global loads per point: fine for the two or three points most tiles' last run has left, a second for a voxel of a million
// points (a driver that reports invalid returns as zeros puts them all into the voxel at the origin). After CE_TAIL_INLINE
// points the thread hands the run over (TailRun in shared memory) and the whole CTA finishes it at the end of the tile:
// rounds of CE_TAIL_ITEMS sorted items -- every thread tests its items' keys and fetches the matching points into shared
// memory, all loads in flight together; the run ends at the first item that does not match; one thread extends the sum over
// the matched prefix, in the same strictly sequential order. Not inlined, and fed from a shared-memory copy of the launch
// parameters: the per-voxel code of the kernel keeps its registers and its instruction footprint.
constexpr uint32_t CE_TAIL_INLINE = 24;
constexpr int CE_TAIL_U = 4;
constexpr int CE_TAIL_ITEMS = CE_TAIL_U * VX_THREADS;
struct TailRun {
  float sx, sy, sz, sw;
  unsigned long long key;  // the logical key (frame bits included)
  uint32_t n, dst, g;      // points summed so far, index of the voxel in the dense output, first sorted position not yet summed
  uint32_t count_frame;    // 1: the voxel still has to be counted for its frame
};
template <typename KeyT, bool SEG>
__device__ __noinline__ void finish_tail_run(const VoxelParams* pp, const TailRun* tr_s, float4* s_pts, uint32_t* s_lead) {
  constexpr bool REC = SEG || sizeof(KeyT) == 4;
  const VoxelParams& p = *pp;
  const TailRun tr = *tr_s;
  const uint32_t tid = threadIdx.x, lane = tid & 31u;
  const SortInfo si = *p.info;
  const uint32_t F = p.n_frames, idx_bits = si.idx_bits;
  const bool odd = (si.num_passes & 1u) != 0u;
  const void* __restrict__ sorted = odd ? p.keys_b : p.keys_a;
  const uint32_t* __restrict__ vals = odd ? p.vals_b : p.vals_a;
  // the sorted keys that continue the run: the key itself; for frame-segmented runs the bare index, inside the frame's range
  uint32_t limit = p.frame_surv_start[F];
  unsigned long long want = tr.key;
  if (SEG) {
    limit = p.frame_surv_start[(tr.key >> idx_bits) + 1ull];
    want = tr.key & ((1ull << idx_bits) - 1ull);
  }
  float sx = tr.sx, sy = tr.sy, sz = tr.sz, sw = tr.sw;
  uint32_t n = tr.n, g = tr.g;
  while (true) {
#pragma unroll 1
    for (int u = 0; u < CE_TAIL_U; ++u) {
      const uint32_t i = g + (uint32_t)u * VX_THREADS + tid;
      bool m = i < limit && i >= g;
      uint32_t slot = 0;
      if (m) {
        if (REC) {
          const uint2 r = reinterpret_cast<const uint2*>(sorted)[i];
          m = (unsigned long long)r.x == want;
          slot = r.y;
        } else {
          m = (unsigned long long)reinterpret_cast<const KeyT*>(sorted)[i] == want;
          slot = vals[i];
        }
      }
      const uint32_t bal = __ballot_sync(0xFFFFFFFFu, m);
      if (lane == 0) s_lead[u * (VX_THREADS / 32) + (tid >> 5)] = bal == 0xFFFFFFFFu ? 32u : (uint32_t)__ffs(~bal) - 1u;
      if (m) s_pts[u * VX_THREADS + tid] = __ldg(p.pts + slot);
    }
    __syncthreads();
    uint32_t matched = 0;
    bool open = true;
#pragma unroll 1
    for (int w = 0; w < CE_TAIL_U * (VX_THREADS / 32); ++w) {
      const uint32_t l = s_lead[w];
      matched += open ? l : 0u;
      open = open && l == 32u;
    }
    if (tid == 0) {
      for (uint32_t q = 0; q < matched; ++q) {
        const float4 pt = s_pts[q];
        sx = __fadd_rn(sx, pt.x); sy = __fadd_rn(sy, pt.y); sz = __fadd_rn(sz, pt.z); sw = __fadd_rn(sw, pt.w);
      }
    }
    n += matched;
    g += matched;
    __syncthreads();  // s_pts and s_lead are rewritten by the next round
    if (matched < (uint32_t)CE_TAIL_ITEMS) break;
  }
  if (tid == 0) {
    const float nf = (float)n;
    const float4 c = make_float4(__fdiv_rn(sx, nf), __fdiv_rn(sy, nf), __fdiv_rn(sz, nf), p.downsample_all ? __fdiv_rn(sw, nf) : 0.f);
    if (p.out_step == 32) {  // pcl::PointXYZI record: x y z 1.0f | intensity 0 0 0
      float4* o = reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(p.out_xyzi) + (size_t)tr.dst * 32);
      o[0] = make_float4(c.x, c.y, c.z, 1.0f);
      o[1] = make_float4(c.w, 0.f, 0.f, 0.f);
    } else {
      reinterpret_cast<float4*>(p.out_xyzi)[tr.dst] = c;
    }
    p.out_count[tr.dst] = n;
    const unsigned long long f = idx_bits >= 64 ? 0ull : tr.key >> idx_bits;
    unsigned long long vidx = idx_bits >= 64 ? tr.key : tr.key & ((1ull << idx_bits) - 1ull);
    if (p.fused_keys) {  // box-grid index -> PCL's idx on the frame's data-derived grid (as in the kernel's emit)
      const uint32_t b = (uint32_t)vidx;
      const uint32_t k2 = b / p.box.mul2, r2 = b - k2 * p.box.mul2;
      const uint32_t k1 = r2 / p.box.mul1, k0 = r2 - k1 * p.box.mul1;
      const GridDev* __restrict__ gd = p.grid + (f < F ? f : 0ull);
      const long long c0 = (long long)k0 + p.box.min_b[0] - gd->min_b[0];
      const long long c1 = (long long)k1 + p.box.min_b[1] - gd->min_b[1];
      const long long c2 = (long long)k2 + p.box.min_b[2] - gd->min_b[2];
      vidx = (unsigned long long)(c0 + c1 * (long long)gd->mul1 + c2 * (long long)gd->mul2);
    }
    p.out_idx[tr.dst] = vidx;
    if (tr.count_frame && f < F) atomicAdd(&p.acc[f].voxel_count, 1u);
  }
}

constexpr uint32_t CE_SEG_SMEM_FRAMES = 256;  // frame starts staged in shared memory up to here (else read from L2)
template <typename KeyT, bool SEG = false>
__global__ void __launch_bounds__(VX_THREADS, CE_MIN_CTAS) k_voxel_centroid(const VoxelParams p) {
  static_assert(!SEG || sizeof(KeyT) == 8, "the logical key of a segmented run is 64 bits wide");
  constexpr bool REC = SEG || sizeof(KeyT) == 4;  // 8-byte (key, value) records
  __shared__ uint32_t s_fss[SEG ? CE_SEG_SMEM_FRAMES + 1 : 1];
  __shared__ uint32_t s_scan[9];
  extern __shared__ __align__(16) float4 s_pts_buf[];  // CE_PT_BUFS point buffers of CE_TILE (CE_DYN_SMEM bytes)
  __shared__ uint32_t s_headw[CE_TILE / 32 + 1];  // bit i: item i starts a run; bit tile_n: sentinel
  __shared__ unsigned short s_start[CE_TILE];     // tile-local position of the r-th surviving run
  __shared__ uint32_t s_tile, s_base;
  __shared__ uint32_t s_cnt8[VX_THREADS / 32];
  __shared__ VoxelParams s_params;  // for finish_tail_run (a kernel parameter has no address a call could take cheaply)
  __shared__ TailRun s_tail;
  __shared__ uint32_t s_tail_r;     // which run of the tile was handed over (0xFFFFFFFF: none)
  __shared__ uint32_t s_tail_lead[CE_TAIL_U * (VX_THREADS / 32)];
  const uint32_t tid = threadIdx.x, lane = tid & 31u;
  const uint32_t F = p.n_frames;
  const uint32_t M = p.frame_surv_start[F];
  const uint32_t n_tiles = (M + CE_TILE - 1) / CE_TILE;
  if (p.dual_width && ((p.info->width == 4u) != REC)) return;  // the other key width runs
  if (SEG != (p.info->segmented != 0u)) return;
  // Persistent CTAs; tiles are handed out by arrival (a ticket), not by block index: the dense output position of a tile's
  // voxels comes from a look-back over the tiles before it, and a tile may only wait for tiles that are already running or
  // done.
  if (tid == 0) s_tile = atomicAdd(&p.ctrl->cent_ticket, 1u);
  __syncthreads();
  uint32_t tile = s_tile;
  if (tile >= n_tiles) return;
  for (uint32_t i = tid; i < sizeof(VoxelParams) / 4; i += VX_THREADS)
    reinterpret_cast<uint32_t*>(&s_params)[i] = reinterpret_cast<const uint32_t*>(&p)[i];

  const SortInfo si = *p.info;
  const uint32_t idx_bits = si.idx_bits;
  const bool odd = (si.num_passes & 1u) != 0u;
  const uint32_t epoch = *p.epoch_dev + 9u;  // the radix passes of this run use + 1 .. + 8
  // 32-bit keys arrive as 8-byte (key, value) records, 64-bit keys as two arrays
  const void* __restrict__ sorted = odd ? p.keys_b : p.keys_a;
  const uint32_t* __restrict__ vals = odd ? p.vals_b : p.vals_a;
  // SEG: start of frame f / the last frame that starts at or before position i (empty frames in front of it are skipped)
  const bool fss_staged = SEG && F <= CE_SEG_SMEM_FRAMES;
  if (fss_staged) {
    for (uint32_t i = tid; i <= F; i += VX_THREADS) s_fss[i] = p.frame_surv_start[i];
    __syncthreads();
  }
  auto fss_at = [&](uint32_t f) -> uint32_t { return fss_staged ? s_fss[f] : p.frame_surv_start[f]; };
  auto frame_between = [&](uint32_t i, uint32_t lo, uint32_t hi) -> uint32_t {
    while (lo < hi) {
      const uint32_t mid = (lo + hi + 1u) >> 1;
      if (fss_at(mid) <= i) lo = mid; else hi = mid - 1u;
    }
    return lo;
  };
  // the frames of the tile the CTA looked at last (item_flags): nearly every tile lies inside one frame, and then nothing is
  // searched for its items
  uint32_t rng_b = 0, rng_e = 0, rng_lo = 0, rng_hi = 0;
  auto frame_of = [&](uint32_t i) -> uint32_t {
    if (i >= rng_b && i < rng_e) return rng_lo == rng_hi ? rng_lo : frame_between(i, rng_lo, rng_hi);
    return frame_between(i, 0u, F - 1u);
  };
  auto key_at = [&](uint32_t i) -> KeyT {
    if constexpr (SEG) return ((KeyT)frame_of(i) << idx_bits) | (KeyT) reinterpret_cast<const uint2*>(sorted)[i].x;
    else if constexpr (REC) return (KeyT) reinterpret_cast<const uint2*>(sorted)[i].x;
    else return reinterpret_cast<const KeyT*>(sorted)[i];
  };
  auto val_at = [&](uint32_t i) -> uint32_t {
    if constexpr (REC) return reinterpret_cast<const uint2*>(sorted)[i].y;
    else return vals[i];
  };
  const bool has_sentinel = si.key_frames > F;  // non-finite points were keyed into an extra frame: never emitted
  const unsigned long long limit = (unsigned long long)F << idx_bits;
  const unsigned long long idx_mask = idx_bits >= 64 ? ~0ull : ((1ull << idx_bits) - 1ull);
  const uint32_t m_req = p.min_points > 1u ? p.min_points : 1u;

  const uint32_t loc = tid * CE_IPT;  // tile-local index of this thread's first item

  // SEG: the frames of the tile at tile_base (k_grid_setup's seg_cent_range), for frame_of
  auto frame_range = [&](uint32_t tile_base) {
    rng_b = tile_base;
    rng_e = min(tile_base + (uint32_t)CE_TILE, M);
    const uint2 fr = __ldg(p.seg_cent_range + tile_base / CE_TILE);  // the same in every thread
    rng_lo = fr.x;
    rng_hi = fr.y;
  };

  // keys (and point slots) of this thread's eight items of the tile at tile_base, and what they say about runs:
  //   head bit j: item j starts a run; pass bit j: ... a run that survives the min-points filter; need bit j: its point is summed
  auto item_flags = [&](uint32_t tile_base, KeyT (&k)[CE_IPT], uint32_t (&v)[CE_IPT], bool want_vals, uint32_t& head, uint32_t& pass,
                        uint32_t& need) {
    const uint32_t base = tile_base + loc;
    if (base + CE_IPT <= M) {
      if constexpr (REC) {
        const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const uint2*>(sorted) + base);
#pragma unroll
        for (int j = 0; j < CE_IPT; j += 2) {
          const uint4 r = src[j / 2];
          k[j] = (KeyT)r.x; v[j] = r.y; k[j + 1] = (KeyT)r.z; v[j + 1] = r.w;
        }
      } else {
        const ulonglong2* ks = reinterpret_cast<const ulonglong2*>(reinterpret_cast<const KeyT*>(sorted) + base);
#pragma unroll
        for (int j = 0; j < CE_IPT; j += 2) {
          const ulonglong2 r = ks[j / 2];
          k[j] = (KeyT)r.x; k[j + 1] = (KeyT)r.y;
        }
        if (want_vals) {
          const uint4* vs = reinterpret_cast<const uint4*>(vals + base);
#pragma unroll
          for (int j = 0; j < CE_IPT; j += 4) {
            const uint4 r = vs[j / 4];
            v[j] = r.x; v[j + 1] = r.y; v[j + 2] = r.z; v[j + 3] = r.w;
          }
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < CE_IPT; ++j) {
        const bool in = base + j < M;
        if constexpr (SEG) k[j] = in ? (KeyT) reinterpret_cast<const uint2*>(sorted)[base + j].x : (KeyT)0;
        else k[j] = in ? key_at(base + j) : (KeyT)0;
        v[j] = (in && want_vals) ? val_at(base + j) : 0u;
      }
    }
    if constexpr (SEG) {  // frame bits from the position
      frame_range(tile_base);
      if (rng_lo == rng_hi) {
        const KeyT fb = (KeyT)rng_lo << idx_bits;
#pragma unroll
        for (int j = 0; j < CE_IPT; ++j)
          if (base + j < M) k[j] |= fb;
      } else if (base < M) {  // a frame boundary inside the tile: one search for the first item, then forward
        uint32_t f = frame_between(base, rng_lo, rng_hi);
#pragma unroll
        for (int j = 0; j < CE_IPT; ++j) {
          while (f < rng_hi && fss_at(f + 1u) <= base + j) ++f;
          if (base + j < M) k[j] |= (KeyT)f << idx_bits;
        }
      }
    }
    // keys of the items just before and just after this thread's eight
    KeyT prev = (KeyT)__shfl_up_sync(0xFFFFFFFFu, k[CE_IPT - 1], 1);
    KeyT next = (KeyT)__shfl_down_sync(0xFFFFFFFFu, k[0], 1);
    if (lane == 0 && base > 0 && base < M) prev = key_at(base - 1);
    if (lane == 31 && base + CE_IPT < M) next = key_at(base + CE_IPT);
    // eq bit j: item j exists and continues the run of item j-1 (bit CE_IPT: the item after this thread's last)
    uint32_t eq = 0, valid = 0;
#pragma unroll
    for (int j = 0; j < CE_IPT; ++j) {
      const bool in = base + j < M;
      const KeyT before = j == 0 ? prev : k[j - 1];
      valid |= (in ? 1u : 0u) << j;
      eq |= ((in && (base + j > 0) && k[j] == before) ? 1u : 0u) << j;
    }
    eq |= ((base + CE_IPT < M && next == k[CE_IPT - 1]) ? 1u : 0u) << CE_IPT;
    head = valid & ~eq;  // bits 0..7
    // which heads survive the min-points filter, and which points are therefore needed
    pass = head; need = valid;
    if (m_req == 2u) {
      pass = head & (eq >> 1);          // the next item continues the run
      need = valid & (eq | (eq >> 1));  // the item has an equal neighbour
    } else if (m_req > 2u) {
      pass = 0;
#pragma unroll
      for (int j = 0; j < CE_IPT; ++j) {
        if (head & (1u << j)) {
          const unsigned long long i2 = (unsigned long long)base + j + m_req - 1ull;
          if (i2 < (unsigned long long)M && key_at((uint32_t)i2) == k[j]) pass |= 1u << j;
        }
      }
    }
    if (has_sentinel) {
#pragma unroll
      for (int j = 0; j < CE_IPT; ++j)
        if ((unsigned long long)k[j] >= limit) pass &= ~(1u << j);
    }
  };

  // The voxel count of a tile, published the moment the tile is claimed -- a whole tile-time before any later tile looks for
  // it: the CTA counts its NEXT tile (keys only: one coalesced sweep, no point gathers) before it works on the current one.
  // With the counts that early, the look-back further down never waits for a tile that is still busy; without this, every tile
  // stalled for the slowest of its ~600 co-resident predecessors and the launch took 0.18 ms instead of 0.12 (measured).
  // The sweep keeps the tile's head and pass bits (registers of the same thread, which owns the same items then) and starts
  // the copies of its needed points into the tile's point buffer, one cp.async group per tile: they land while the CTA works
  // on the current tile, and the tile's own item phase reads neither records nor points from global memory.
  // (CE_PREFETCH, synchronous gathers only: the sweep asks L2 for the points instead; measured, it does not pay -- see the macro.)
  auto count_and_publish = [&](uint32_t t, float4* pts_dst, uint32_t& head, uint32_t& pass) {
    KeyT k[CE_IPT];
    uint32_t v[CE_IPT];
    uint32_t need;
    item_flags(t * CE_TILE, k, v, CE_ASYNC_GATHER || CE_PREFETCH, head, pass, need);
#if CE_ASYNC_GATHER
#pragma unroll
    for (int j = 0; j < CE_IPT; ++j)
      if (need & (1u << j)) cp_async_16(pts_dst + loc + j, p.pts + v[j]);
    cp_async_commit();
#elif CE_PREFETCH
#pragma unroll
    for (int j = 0; j < CE_IPT; ++j)
      if (need & (1u << j)) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.pts + v[j]));
#endif
    const uint32_t wsum = warp_sum_u32((uint32_t)__popc(pass));
    // s_cnt8 is this lambda's own scratch: its previous use lies a whole tile (several barriers) back
    if (lane == 0) s_cnt8[tid >> 5] = wsum;
    __syncthreads();
    if (tid == 0) {
      uint32_t tot = 0;
#pragma unroll
      for (int w = 0; w < VX_THREADS / 32; ++w) tot += s_cnt8[w];
      st_relaxed_u64(p.cent_status + t, lb_pack(epoch, t == 0u ? CM_LB_INCL : CM_LB_AGG, tot));
    }
  };

  uint32_t head, pass;  // this thread's flags of `tile`, from its count sweep
  uint32_t buf = 0;     // which point buffer holds `tile`'s points
  count_and_publish(tile, s_pts_buf, head, pass);
  while (true) {
  // claim and count the next tile first
  if (tid == 0) s_tile = atomicAdd(&p.ctrl->cent_ticket, 1u);
  __syncthreads();  // also: the last reads of the other point buffer (the previous tile) are done
  const uint32_t next_tile = s_tile;
  const uint32_t next_buf = (buf + 1u) % CE_PT_BUFS;
  uint32_t next_head = 0, next_pass = 0;
  if (next_tile < n_tiles) count_and_publish(next_tile, s_pts_buf + next_buf * CE_TILE, next_head, next_pass);

  const uint32_t tile_base = tile * CE_TILE;
  const uint32_t tile_n = min((uint32_t)CE_TILE, M - tile_base);
  float4* const s_pts = s_pts_buf + buf * CE_TILE;

  // ---- per item -----------------------------------------------------------------------------------------------------
#if CE_ASYNC_GATHER
  // this thread's copies of the tile are in (the next tile's group may still fly); the scan's barrier shows them to the CTA.
  // Without a next tile nothing is left in flight.
  if (next_tile < n_tiles) cp_async_wait<1>();
  else cp_async_wait<0>();
  if constexpr (SEG) frame_range(tile_base);  // the sweep left the next tile's frames behind
#else
  {
    KeyT k[CE_IPT];
    uint32_t v[CE_IPT];
    uint32_t need;
    item_flags(tile_base, k, v, true, head, pass, need);
#pragma unroll
    for (int j = 0; j < CE_IPT; ++j)
      if (need & (1u << j)) s_pts[loc + j] = __ldg(p.pts + v[j]);
  }
#endif
  reinterpret_cast<unsigned char*>(s_headw)[tid] = (unsigned char)head;  // bit position 8*tid + j == item loc + j
  if (tid == 0) { s_headw[CE_TILE / 32] = 0u; s_tail_r = 0xFFFFFFFFu; }
  const uint32_t cnt = (uint32_t)__popc(pass);

  uint32_t total;
  const uint32_t excl_thread = block_excl_scan_256(cnt, s_scan, &total);  // also orders the shared-memory staging
  {
    uint32_t r = excl_thread, pm = pass;
    while (pm) {
      const uint32_t j = (uint32_t)__ffs(pm) - 1u;
      pm &= pm - 1u;
      s_start[r++] = (unsigned short)(loc + j);
    }
    if (tid == 0) {
      atomicOr(&s_headw[tile_n >> 5], 1u << (tile_n & 31u));  // sentinel: every run ends at the end of the tile at the latest
    }
  }
  __syncthreads();

  // ---- dense output position of this tile's first voxel: decoupled look-back, one warp, 32 earlier tiles per round (lane l
  // looks at tile j - l). The other warps go on to their first voxel and meet this one at the barrier before the stores.
  if (tid < 32) {
    uint32_t base = 0;
#ifdef CE_DEBUG_NO_LOOKBACK   // timing experiment only (wrong output positions): what the kernel costs without the chain
    if (false) {
#else
    if (tile > 0) {
#endif
      long long j = (long long)tile - 1;  // newest tile of the window
      uint32_t spins = 0;
      unsigned long long wd0 = 0ull;
      while (true) {
        const long long t = j - (long long)lane;
        // tiles before the first one: an inclusive prefix of zero
        const unsigned long long w = t >= 0 ? ld_cg_u64(p.cent_status + t) : lb_pack(epoch, CM_LB_INCL, 0u);
        const uint32_t hi = (uint32_t)(w >> 32);
        const bool ready = (hi >> 2) == epoch && (hi & 3u) != 0u;
        const uint32_t not_ready = __ballot_sync(0xFFFFFFFFu, !ready);
        if (not_ready) {
#if CE_LB_POLL_ONE
          // wait on the nearest unpublished word with ONE lane, then read the window again
          const long long wait_for = j - (long long)(__ffs(not_ready) - 1);
          bool expired = false;
          if (lane == 0) {
            while (true) {
              const unsigned long long x = ld_relaxed_u64(p.cent_status + wait_for);
              const uint32_t xh = (uint32_t)(x >> 32);
              if ((xh >> 2) == epoch && (xh & 3u) != 0u) break;
              if (watchdog_expired(spins, wd0)) { expired = true; break; }
              __nanosleep(CE_LB_POLL_NS);
            }
          }
          if (__any_sync(0xFFFFFFFFu, expired)) {
            atomicExch(&p.ctrl->error, (uint32_t)CM_DEV_E_INTERNAL);
            break;
          }
#else
          if (__any_sync(0xFFFFFFFFu, watchdog_expired(spins, wd0))) {
            atomicExch(&p.ctrl->error, (uint32_t)CM_DEV_E_INTERNAL);
            break;
          }
          if (spins > 4) __nanosleep(CE_LB_POLL_NS);
#endif
          continue;
        }
        const uint32_t incl = __ballot_sync(0xFFFFFFFFu, (hi & 3u) == CM_LB_INCL);
        const uint32_t stop = incl ? (uint32_t)__ffs(incl) - 1u : 32u;  // nearest tile that already knows its inclusive prefix
        base += warp_sum_u32(lane <= stop ? (uint32_t)w : 0u);
        if (incl) break;
        j -= 32;
      }
      if (lane == 0) st_relaxed_u64(p.cent_status + tile, lb_pack(epoch, CM_LB_INCL, base + total));
    }
    if (lane == 0) {
      s_base = base;
      if (tile == n_tiles - 1u) p.ctrl->total_voxels = base + total;
    }
  }

  // per-frame voxel counts: one atomic per tile unless the tile straddles frames
  bool per_voxel_count = false;
  if (F == 1) {
    if (tid == 0 && total) atomicAdd(&p.acc[0].voxel_count, total);
  } else {
    const unsigned long long f_first = (unsigned long long)key_at(tile_base) >> idx_bits;
    const unsigned long long f_last = (unsigned long long)key_at(tile_base + tile_n - 1) >> idx_bits;
    if (f_first == f_last) {
      if (tid == 0 && total && f_first < F) atomicAdd(&p.acc[f_first].voxel_count, total);
    } else {
      per_voxel_count = true;
    }
  }

  // ---- per voxel ----------------------------------------------------------------------------------------------------
  // The first voxel of every thread is summed BEFORE the barrier that delivers the tile's output position, so the look-back
  // of warp 0 hides behind it; further voxels (tiles with more than 256 surviving runs) follow after the barrier.
  // false: the run was handed over to the CTA (tail run) -- nothing to emit here
  auto voxel = [&](uint32_t r, float4& cen, uint32_t& n_out, KeyT& key_out) -> bool {
    const uint32_t s0 = s_start[r];
    const KeyT key = key_at(tile_base + s0);
    // end of the run inside the tile: the next head bit after s0 (the sentinel at tile_n bounds the search)
    uint32_t q = s0 + 1u;
    uint32_t w = q >> 5;
    uint32_t bits = s_headw[w] & (0xFFFFFFFFu << (q & 31u));
    while (bits == 0u) bits = s_headw[++w];
    const uint32_t end = (w << 5) + (uint32_t)__ffs(bits) - 1u;
    float sx = 0.f, sy = 0.f, sz = 0.f, sw = 0.f;
    for (q = s0; q < end; ++q) {
      const float4 pt = s_pts[q];
      sx = __fadd_rn(sx, pt.x); sy = __fadd_rn(sy, pt.y); sz = __fadd_rn(sz, pt.z); sw = __fadd_rn(sw, pt.w);
    }
    uint32_t n = end - s0;
    if (end == tile_n) {  // the run may continue in the following tiles: global memory
      uint32_t g = tile_base + tile_n;
      while (g < M && key_at(g) == key) {
        if (g - (tile_base + tile_n) == CE_TAIL_INLINE) {  // a long run: the CTA finishes it (finish_tail_run)
          s_tail.sx = sx; s_tail.sy = sy; s_tail.sz = sz; s_tail.sw = sw;
          s_tail.key = (unsigned long long)key; s_tail.n = n; s_tail.g = g;
          s_tail_r = r;
          return false;
        }
        const float4 pt = __ldg(p.pts + val_at(g));
        sx = __fadd_rn(sx, pt.x); sy = __fadd_rn(sy, pt.y); sz = __fadd_rn(sz, pt.z); sw = __fadd_rn(sw, pt.w);
        ++n; ++g;
      }
    }
    if (n == 1u) {  // x / 1.0f == x: a voxel of one point (most voxels of a fine leaf) needs no division
      cen = make_float4(sx, sy, sz, p.downsample_all ? sw : 0.f);
    } else {
      const float nf = (float)n;
      cen = make_float4(__fdiv_rn(sx, nf), __fdiv_rn(sy, nf), __fdiv_rn(sz, nf), p.downsample_all ? __fdiv_rn(sw, nf) : 0.f);
    }
    n_out = n;
    key_out = key;
    return true;
  };
  auto emit = [&](uint32_t dst, const float4& c, uint32_t n, KeyT key) {
    if (p.out_step == 32) {  // pcl::PointXYZI record: x y z 1.0f | intensity 0 0 0
      float4* o = reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(p.out_xyzi) + (size_t)dst * 32);
      o[0] = make_float4(c.x, c.y, c.z, 1.0f);
      o[1] = make_float4(c.w, 0.f, 0.f, 0.f);
    } else {
      reinterpret_cast<float4*>(p.out_xyzi)[dst] = c;
    }
    p.out_count[dst] = n;
    unsigned long long vidx = (unsigned long long)key & idx_mask;
    if (p.fused_keys) {
      // the key indexes the crop box's grid: back to PCL's idx on the frame's data-derived grid (same cells, other origin)
      const uint32_t b = (uint32_t)vidx;
      const uint32_t k2 = b / p.box.mul2, r2 = b - k2 * p.box.mul2;
      const uint32_t k1 = r2 / p.box.mul1, k0 = r2 - k1 * p.box.mul1;
      const unsigned long long f = (unsigned long long)key >> idx_bits;
      const GridDev* __restrict__ g = p.grid + (f < F ? f : 0ull);
      const long long c0 = (long long)k0 + p.box.min_b[0] - g->min_b[0];
      const long long c1 = (long long)k1 + p.box.min_b[1] - g->min_b[1];
      const long long c2 = (long long)k2 + p.box.min_b[2] - g->min_b[2];
      vidx = (unsigned long long)(c0 + c1 * (long long)g->mul1 + c2 * (long long)g->mul2);
    }
    p.out_idx[dst] = vidx;
    if (per_voxel_count) {
      const unsigned long long f = (unsigned long long)key >> idx_bits;
      if (f < F) atomicAdd(&p.acc[f].voxel_count, 1u);
    }
  };
  float4 c0 = make_float4(0.f, 0.f, 0.f, 0.f);
  uint32_t n0 = 0;
  KeyT k0 = (KeyT)0;
  bool whole0 = false;
  if (tid < total) whole0 = voxel(tid, c0, n0, k0);
  __syncthreads();  // s_base: the look-back of warp 0 is done
  const uint32_t out0 = s_base;
  if (whole0) emit(out0 + tid, c0, n0, k0);
  for (uint32_t r = tid + VX_THREADS; r < total; r += VX_THREADS)
    if (voxel(r, c0, n0, k0)) emit(out0 + r, c0, n0, k0);
  __syncthreads();  // every read of this tile's shared memory is done
  if (s_tail_r != 0xFFFFFFFFu) {  // (block-uniform) at most one run per tile is handed over
    if (tid == 0) {
      s_tail.dst = out0 + s_tail_r;
      s_tail.count_frame = per_voxel_count ? 1u : 0u;
    }
    __syncthreads();
    finish_tail_run<KeyT, SEG>(&s_params, &s_tail, s_pts, s_tail_lead);  // scratch: this tile's buffer, not the one in flight
    __syncthreads();
  }
  tile = next_tile;
  head = next_head;
  pass = next_pass;
  buf = next_buf;
  if (tile >= n_tiles) break;
  }  // while (true): next tile
}

// ---- host path: the frame's dense voxel outputs -> page-locked (device-mapped) host memory ------------------------------
// Last kernel of a host-path frame. The number of voxels is only known on the device (Ctrl.total_voxels), so a
// cudaMemcpyAsync of the right size would need a host round trip first; this kernel reads the count itself and pushes the
// three arrays over PCIe with 16-byte stores (a frame's voxels are ~1 MB: a few microseconds of link time).
__global__ void __launch_bounds__(VX_THREADS) k_export_voxels(const VoxelParams p, uint4* __restrict__ host_xyzi,
                                                             uint32_t* __restrict__ host_count,
                                                             unsigned long long* __restrict__ host_idx, uint32_t cap) {
  const uint32_t V = min(p.ctrl->total_voxels, cap);
  const uint32_t stride = gridDim.x * VX_THREADS, t0 = blockIdx.x * VX_THREADS + threadIdx.x;
  const uint32_t n16 = V * (p.out_step / 16u);
  const uint4* __restrict__ sx = reinterpret_cast<const uint4*>(p.out_xyzi);
  for (uint32_t i = t0; i < n16; i += stride) host_xyzi[i] = sx[i];
  const uint4* __restrict__ sc = reinterpret_cast<const uint4*>(p.out_count);
  for (uint32_t i = t0; i < V / 4u; i += stride) reinterpret_cast<uint4*>(host_count)[i] = sc[i];
  const uint4* __restrict__ si = reinterpret_cast<const uint4*>(p.out_idx);
  for (uint32_t i = t0; i < V / 2u; i += stride) reinterpret_cast<uint4*>(host_idx)[i] = si[i];
  if (blockIdx.x == 0) {  // tails
    for (uint32_t i = (V & ~3u) + threadIdx.x; i < V; i += VX_THREADS) host_count[i] = p.out_count[i];
    for (uint32_t i = (V & ~1u) + threadIdx.x; i < V; i += VX_THREADS) host_idx[i] = p.out_idx[i];
  }
}

// ---- launchers ----------------------------------------------------------------------------------------------------
static inline uint32_t persistent_grid(uint32_t n_tiles) {
  const uint32_t cap = 148u * 8u;
  return n_tiles < 1u ? 1u : (n_tiles < cap ? n_tiles : cap);
}

cudaError_t launch_minmax(const float4* pts, uint32_t n, Ctrl* ctrl, FrameAcc* acc, uint32_t* frame_surv_start,
                          cudaStream_t stream) {
  const uint32_t tiles = (n + KH_TILE - 1) / KH_TILE;
  k_minmax<<<persistent_grid(tiles), VX_THREADS, 0, stream>>>(pts, n, ctrl, acc, frame_surv_start);
  return cudaGetLastError();
}

cudaError_t launch_seed_bounds(FrameAcc* acc, const float* mn, const float* mx, cudaStream_t stream) {
  k_seed_bounds<<<1, 32, 0, stream>>>(acc, mn[0], mn[1], mn[2], mx[0], mx[1], mx[2]);
  return cudaGetLastError();
}

cudaError_t launch_tile_scan(TileRec* tile_rec, uint32_t n_tiles, const SegDev* segs, uint32_t n_seg, uint32_t n_frames,
                             uint32_t* frame_surv_start, uint32_t* seg_surv_start, cudaStream_t stream) {
  k_tile_scan<<<1, SCAN_THREADS, 0, stream>>>(tile_rec, n_tiles, segs, n_seg, n_frames, frame_surv_start, seg_surv_start);
  return cudaGetLastError();
}

cudaError_t launch_compact_survivors(const TileRec* tile_rec, uint32_t n_tiles, const float4* slot_xyzi,
                                     const uint32_t* slot_src, float4* dense_xyzi, uint32_t* dense_src,
                                     uint32_t* dense_slot, cudaStream_t stream) {
  if (n_tiles == 0) return cudaSuccess;
  k_compact_survivors<<<persistent_grid(n_tiles), VX_THREADS, 0, stream>>>(tile_rec, n_tiles, slot_xyzi, slot_src,
                                                                            dense_xyzi, dense_src, dense_slot);
  return cudaGetLastError();
}

cudaError_t launch_grid_setup(const VoxelParams& p, cudaStream_t stream, TileRec* scan_rec, uint32_t scan_tiles,
                              const SegDev* segs, uint32_t n_seg, uint32_t* seg_surv_start) {
  TileScanArgs ts;
  ts.rec = scan_rec; ts.n_tiles = scan_tiles; ts.segs = segs; ts.n_seg = n_seg; ts.seg_surv_start = seg_surv_start;
  k_grid_setup<<<1, SCAN_THREADS, 0, stream>>>(p, ts);
  return cudaGetLastError();
}

cudaError_t launch_key_hist(const VoxelParams& p, cudaStream_t stream) {
  const uint32_t tiles = p.tile_rec ? p.n_k1_tiles : (p.max_points + KH_DENSE_TILE - 1) / KH_DENSE_TILE + p.n_frames;
  if (p.key_bytes == 4)
    k_voxel_key_hist<uint32_t><<<persistent_grid(tiles), VX_THREADS, 0, stream>>>(p);
  else
    k_voxel_key_hist<unsigned long long><<<persistent_grid(tiles), VX_THREADS, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_seg_base(const VoxelParams& p, cudaStream_t stream) {
  if (p.n_frames == 0) return cudaSuccess;
  if (p.fused_keys && p.box.seg_sort)
    k_seg_base<CM_WIDE_BINS><<<dim3(p.n_frames, CM_SEG_PASSES), CM_WIDE_BINS, 0, stream>>>(p);
  else
    k_seg_base<CM_RADIX><<<dim3(p.n_frames, CM_SEG_PASSES), CM_RADIX, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_seg_keys64(const void* records, unsigned long long* keys, uint32_t* vals, const VoxelParams& p,
                              cudaStream_t stream) {
  if (p.max_points == 0) return cudaSuccess;
  const uint32_t blocks = std::min<uint32_t>((p.max_points + VX_THREADS - 1u) / VX_THREADS, 148u * 8u);
  k_seg_keys64<<<blocks, VX_THREADS, 0, stream>>>(reinterpret_cast<const uint2*>(records), keys, vals, p);
  return cudaGetLastError();
}

cudaError_t launch_centroid(const VoxelParams& p, cudaStream_t stream) {
  const uint32_t tiles = (p.max_points + CE_TILE - 1) / CE_TILE;
  if (tiles == 0) return cudaSuccess;
  // persistent: what the device holds at once (tiles are handed out by a ticket)
  const uint32_t grid = std::min<uint32_t>(tiles, 148u * (uint32_t)CE_MIN_CTAS);
  if (p.key_bytes == 4 && p.segmented)
    k_voxel_centroid<unsigned long long, true><<<grid, VX_THREADS, CE_DYN_SMEM, stream>>>(p);
  else if (p.key_bytes == 4)
    k_voxel_centroid<uint32_t><<<grid, VX_THREADS, CE_DYN_SMEM, stream>>>(p);
  else
    k_voxel_centroid<unsigned long long><<<grid, VX_THREADS, CE_DYN_SMEM, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t configure_centroid_kernels() {
  cudaError_t e = cudaFuncSetAttribute(k_voxel_centroid<unsigned long long, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)CE_DYN_SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(k_voxel_centroid<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CE_DYN_SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(k_voxel_centroid<unsigned long long>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CE_DYN_SMEM);
  return e;
}

cudaError_t launch_export_voxels(const VoxelParams& p, void* host_xyzi, uint32_t* host_count, unsigned long long* host_idx,
                                 uint32_t cap, cudaStream_t stream) {
  const uint32_t blocks = std::max(1u, std::min<uint32_t>(148u, (cap + 4u * VX_THREADS - 1u) / (4u * VX_THREADS)));
  k_export_voxels<<<blocks, VX_THREADS, 0, stream>>>(p, static_cast<uint4*>(host_xyzi), host_count, host_idx, cap);
  return cudaGetLastError();
}

uint32_t centroid_tile_items() { return CE_TILE; }

}  // namespace cm
