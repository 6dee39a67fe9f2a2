// cm_route.cu -- device side of the single-giant-cloud mode (BASELINE config 4): one cloud block-distributed over the GPUs of
// a box, VoxelGrid with ONE all-to-all that moves every point to the rank owning its voxel-key range.
//
// The reference has no counterpart (one process, one cloud): what is reproduced is the voxel index of PCL 1.8.1
// VoxelGrid::applyFilter (idx = i + j*div_x + k*div_x*div_y with ijk = floor(p * inv_leaf) - min_b, float32 multiply) on the
// GLOBAL grid, because a voxel must not straddle ranks and the concatenation of the rank outputs must be the PCL order.
//   k_route_hist : coarse histogram of the voxel indices (bins of equal key width) -> all-reduced by the host layer to
//                  pick balanced splitters
//   k_route_mask : destination rank of every point = number of splitters <= its voxel index, as a one-hot mask for the
//                  zone-slicing count / scan / scatter kernels (cm_zones.cu), which group the points by destination in
//                  source order -- the send buffer of the all-to-all.
// Roofline: HBM, 16 B read per point and kernel (+ 2 B mask written).
#include "cm_kernels.h"

namespace cm {

namespace {

constexpr int RT_THREADS = 256;

// Up to RT_SMEM_BINS bins the histogram is privatised per CTA in shared memory (hardware-aggregated increments) and
// flushed once: a map cloud puts most of its points on a few planes, and 50 M global atomics on those hot bins took
// 4.7 ms; above that size the counters are updated in global memory directly.
constexpr uint32_t RT_SMEM_BINS = 16384;
constexpr int RT_HIST_THREADS = 512;

__global__ void __launch_bounds__(RT_HIST_THREADS) k_route_hist(const float4* __restrict__ pts, uint32_t n, const RouteGrid g,
                                                                unsigned long long width, uint32_t bins,
                                                                unsigned long long* __restrict__ hist, int use_smem) {
  extern __shared__ uint32_t s_bins[];
  if (use_smem) {
    for (uint32_t b = threadIdx.x; b < bins; b += RT_HIST_THREADS) s_bins[b] = 0;
    __syncthreads();
  }
  for (uint32_t i = blockIdx.x * RT_HIST_THREADS + threadIdx.x; i < n; i += gridDim.x * RT_HIST_THREADS) {
    unsigned long long key;
    if (route_key(g, ldg_stream_f4(pts + i), &key)) {
      unsigned long long b = key / width;
      if (b >= bins) b = bins - 1;
      if (use_smem) atomicAdd(&s_bins[(uint32_t)b], 1u);
      else atomicAdd(hist + b, 1ull);
    }
  }
  if (use_smem) {
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < bins; b += RT_HIST_THREADS) {
      const uint32_t c = s_bins[b];
      if (c) atomicAdd(hist + b, (unsigned long long)c);
    }
  }
}

__global__ void __launch_bounds__(RT_THREADS) k_route_mask(const float4* __restrict__ pts, uint32_t n, const RouteGrid g,
                                                           const RouteSplit sp, unsigned short* __restrict__ mask) {
  for (uint32_t i = blockIdx.x * RT_THREADS + threadIdx.x; i < n; i += gridDim.x * RT_THREADS) {
    unsigned long long key;
    uint32_t dest = sp.invalid_part;  // non-finite points stay where they are (VoxelGrid skips them)
    if (route_key(g, ldg_stream_f4(pts + i), &key)) {
      dest = 0;
      for (int k = 0; k < sp.n_parts - 1; ++k) dest += (key >= sp.splitter[k]) ? 1u : 0u;
    }
    mask[i] = (unsigned short)(1u << dest);
  }
}

// ---- the same steps with the plan in device memory (cm_giant_voxelgrid: no host round trip between them) ----------------------
// PCL's grid on the all-reduced bounding box (VoxelGrid::applyFilter, float32): min_b = floor(min_p * inv), div_b = max_b - min_b + 1
__global__ void k_giant_plan(GiantPlan* plan, const FrameAcc* __restrict__ acc, float inv0, float inv1, float inv2, uint32_t bins) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  GiantPlan p;
  const float inv[3] = {inv0, inv1, inv2};
  p.error = 0;
  const bool empty = acc->max_enc[0] == 0u && acc->nmin_enc[0] == 0u;  // no finite point anywhere
  long long div[3] = {1, 1, 1};
  for (int k = 0; k < 3; ++k) {
    p.enc[k] = acc->max_enc[k];
    p.enc[3 + k] = acc->nmin_enc[k];
    p.grid.inv[k] = inv[k];
    p.grid.min_b[k] = 0;
    if (!empty) {
      const float mn = __uint_as_float(f32_order_dec(~acc->nmin_enc[k])), mx = __uint_as_float(f32_order_dec(acc->max_enc[k]));
      const float fmn = floorf(__fmul_rn(mn, inv[k])), fmx = floorf(__fmul_rn(mx, inv[k]));
      if (!(fabsf(fmn) < 1073741824.f) || !(fabsf(fmx) < 1073741824.f) || fmx < fmn) p.error = CM_DEV_E_KEY_RANGE;
      else {
        p.grid.min_b[k] = (long long)fmn;
        div[k] = (long long)fmx - (long long)fmn + 1;
        if (div[k] > (1ll << 21)) { p.error = CM_DEV_E_KEY_RANGE; div[k] = 1; }
      }
    }
    p.min_b[k] = (int32_t)p.grid.min_b[k];
    p.div_b[k] = (int32_t)div[k];
  }
  p.grid.div0 = div[0];
  p.grid.div01 = div[0] * div[1];
  p.cells = (unsigned long long)div[0] * (unsigned long long)div[1] * (unsigned long long)div[2];
  p.width = (p.cells + (unsigned long long)bins - 1ull) / (unsigned long long)bins;
  if (p.width == 0) p.width = 1;
  p.key_bits = p.cells <= 1ull ? 0u : (uint32_t)(64 - __clzll((long long)(p.cells - 1ull)));
  p.total = 0;
  p.n_invalid = acc->n_invalid;  // the all-reduce covers max_enc / nmin_enc only: this is the local count
  for (int r = 0; r < CM_MAX_ZONES; ++r) p.splitter[r] = ~0ull;
  *plan = p;
}

// floor(key / width) without the 64-bit division sequence (~100 instructions per point): the quotient is below 2^15 bins, so the
// double-precision estimate is off by one at most, and one multiply-subtract puts it right. Exactly key / width.
__device__ __forceinline__ unsigned long long div_small_quotient(unsigned long long key, unsigned long long width, double inv_w) {
  unsigned long long q = __double2ull_rz(__ull2double_rn(key) * inv_w);
  const long long r = (long long)(key - q * width);
  if (r < 0) --q;
  else if ((unsigned long long)r >= width) ++q;
  return q;
}

// Four points per thread in flight; one CTA per SM flushes its shared-memory bins once, starting at a bin of its own so that
// the CTAs do not queue up on the same counters.
constexpr int GH_THREADS = 1024;
constexpr int GH_UNROLL = 4;
__global__ void __launch_bounds__(GH_THREADS) k_giant_hist(const float4* __restrict__ pts, uint32_t n,
                                                           const GiantPlan* __restrict__ plan, uint32_t bins,
                                                           unsigned long long* __restrict__ hist, int use_smem) {
  extern __shared__ uint32_t s_bins[];
  const RouteGrid g = plan->grid;
  const unsigned long long width = plan->width;
  const double inv_w = 1.0 / __ull2double_rn(width);
  const bool small_q = plan->cells / width < (1ull << 40);  // always, by the choice of the width; the exact division otherwise
  if (use_smem) {
    for (uint32_t b = threadIdx.x; b < bins; b += GH_THREADS) s_bins[b] = 0;
    __syncthreads();
  }
  const uint32_t stride = gridDim.x * GH_THREADS;
  for (uint32_t i0 = blockIdx.x * GH_THREADS + threadIdx.x; i0 < n; i0 += GH_UNROLL * stride) {
    float4 v[GH_UNROLL];
#pragma unroll
    for (int u = 0; u < GH_UNROLL; ++u) {
      const uint32_t i = i0 + (uint32_t)u * stride;
      v[u] = (i < n && i >= i0) ? ldg_stream_f4(pts + i) : make_float4(__int_as_float(0x7fc00000), 0.f, 0.f, 0.f);  // NaN: skipped
    }
#pragma unroll
    for (int u = 0; u < GH_UNROLL; ++u) {
      unsigned long long key;
      if (route_key(g, v[u], &key)) {
        unsigned long long b = small_q ? div_small_quotient(key, width, inv_w) : key / width;
        if (b >= bins) b = bins - 1;
        if (use_smem) atomicAdd(&s_bins[(uint32_t)b], 1u);
        else atomicAdd(hist + b, 1ull);
      }
    }
  }
  if (use_smem) {
    __syncthreads();
    const uint32_t rot = (uint32_t)(((unsigned long long)blockIdx.x * bins) / gridDim.x);
    for (uint32_t t = threadIdx.x; t < bins; t += GH_THREADS) {
      uint32_t b = t + rot;
      if (b >= bins) b -= bins;
      const uint32_t c = s_bins[b];
      if (c) atomicAdd(hist + b, (unsigned long long)c);
    }
  }
}

// One CTA: running sum of the all-reduced histogram, then the n_parts - 1 splitters that balance the point counts: the first
// bin boundary at or after total * r / n_parts (what pick_splitters of the gloo-tested host protocol computes).
constexpr int GS_THREADS = 1024;
__global__ void __launch_bounds__(GS_THREADS) k_giant_splitters(GiantPlan* plan, const unsigned long long* __restrict__ hist,
                                                                uint32_t bins, uint32_t n_parts) {
  __shared__ unsigned long long s_warp[GS_THREADS / 32];
  __shared__ unsigned long long s_target[CM_MAX_ZONES];
  __shared__ unsigned long long s_total;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t chunk = (bins + GS_THREADS - 1) / GS_THREADS;
  const uint32_t b0 = min(bins, tid * chunk), b1 = min(bins, b0 + chunk);
  // the thread's bins, fetched once with 16-byte loads when the chunk is the usual 16 bins (16 Ki bins / 1024 threads)
  constexpr uint32_t GS_CHUNK = 16;
  unsigned long long hv[GS_CHUNK];
  const bool in_regs = chunk == GS_CHUNK && b1 - b0 == GS_CHUNK;
  if (in_regs) {
    const ulonglong2* src = reinterpret_cast<const ulonglong2*>(hist + b0);
#pragma unroll
    for (uint32_t k = 0; k < GS_CHUNK; k += 2) {
      const ulonglong2 t = src[k / 2];
      hv[k] = t.x; hv[k + 1] = t.y;
    }
  }
  unsigned long long sum = 0;
  if (in_regs) {
#pragma unroll
    for (uint32_t k = 0; k < GS_CHUNK; ++k) sum += hv[k];
  } else {
    for (uint32_t b = b0; b < b1; ++b) sum += hist[b];
  }
  // exclusive scan of the 1024 partial sums: shuffles inside a warp, the 32 warp totals by warp 0
  unsigned long long incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if ((int)lane >= o) incl += t;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const unsigned long long w = s_warp[lane];
    unsigned long long wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, wi, o);
      if ((int)lane >= o) wi += t;
    }
    s_warp[lane] = wi - w;
    if (lane == 31) { s_total = wi; plan->total = wi; }
  }
  __syncthreads();
  const unsigned long long total = s_total, width = plan->width;
  if (tid >= 1 && tid < n_parts) s_target[tid] = total * tid / n_parts;
  __syncthreads();
  // every thread walks its own bins; a target falls into exactly one thread's range of the running sum
  unsigned long long cum = s_warp[warp] + incl - sum;
  auto step = [&](uint32_t b, unsigned long long count) {
    const unsigned long long before = cum;
    cum += count;
    if (cum == before && b != 0) return;  // an empty bin (other than the first) is the first to reach no target
    for (uint32_t r = 1; r < n_parts; ++r) {
      const unsigned long long target = s_target[r];
      // first index i with cum[i] >= target (inclusive running sum), + 1; a target of 0 is met by bin 0
      const bool first = (cum >= target) && (b == 0 ? true : before < target);
      if (first) plan->splitter[r - 1] = (unsigned long long)min(b + 1u, bins) * width;
    }
  };
  if (in_regs) {
#pragma unroll
    for (uint32_t k = 0; k < GS_CHUNK; ++k) step(b0 + k, hv[k]);
  } else {
    for (uint32_t b = b0; b < b1; ++b) step(b, hist[b]);
  }
  if (tid == 0 && total == 0)  // an empty cloud: every splitter at the first boundary (nothing moves)
    for (uint32_t r = 1; r < n_parts; ++r) plan->splitter[r - 1] = width;
}

__global__ void k_seed_bounds_enc(FrameAcc* acc, const uint32_t* __restrict__ enc6) {
  const uint32_t k = threadIdx.x;
  if (blockIdx.x == 0 && k < 6) {
    if (k < 3) atomicMax(&acc->max_enc[k], enc6[k]);
    else atomicMax(&acc->nmin_enc[k - 3], enc6[k]);
  }
}

}  // namespace

cudaError_t launch_giant_plan(GiantPlan* plan, const FrameAcc* acc_reduced, const float* inv_leaf3, uint32_t bins, cudaStream_t stream) {
  k_giant_plan<<<1, 32, 0, stream>>>(plan, acc_reduced, inv_leaf3[0], inv_leaf3[1], inv_leaf3[2], bins);
  return cudaGetLastError();
}

cudaError_t launch_giant_hist(const float4* pts, uint32_t n, const GiantPlan* plan, uint32_t bins, unsigned long long* hist,
                              cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const int use_smem = bins <= RT_SMEM_BINS ? 1 : 0;
  const size_t smem = use_smem ? (size_t)bins * sizeof(uint32_t) : 0;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(k_giant_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(RT_SMEM_BINS * sizeof(uint32_t)));
    if (e != cudaSuccess) return e;
    configured = true;
  }
  const uint32_t blocks = std::min<uint32_t>((n + GH_THREADS * GH_UNROLL - 1) / (GH_THREADS * GH_UNROLL), 148u);
  k_giant_hist<<<blocks, GH_THREADS, smem, stream>>>(pts, n, plan, bins, hist, use_smem);
  return cudaGetLastError();
}

cudaError_t launch_giant_splitters(GiantPlan* plan, const unsigned long long* hist_reduced, uint32_t bins, uint32_t n_parts,
                                   cudaStream_t stream) {
  k_giant_splitters<<<1, GS_THREADS, 0, stream>>>(plan, hist_reduced, bins, n_parts);
  return cudaGetLastError();
}

cudaError_t launch_seed_bounds_enc(FrameAcc* acc, const uint32_t* enc6, cudaStream_t stream) {
  k_seed_bounds_enc<<<1, 32, 0, stream>>>(acc, enc6);
  return cudaGetLastError();
}

cudaError_t launch_route_hist(const float4* pts, uint32_t n, const RouteGrid& g, unsigned long long width, uint32_t bins,
                              unsigned long long* hist, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const int use_smem = bins <= RT_SMEM_BINS ? 1 : 0;
  const size_t smem = use_smem ? (size_t)bins * sizeof(uint32_t) : 0;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(k_route_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(RT_SMEM_BINS * sizeof(uint32_t)));
    if (e != cudaSuccess) return e;
    configured = true;
  }
  const uint32_t blocks = std::min<uint32_t>((n + RT_HIST_THREADS - 1) / RT_HIST_THREADS, 148u * 2u);
  k_route_hist<<<blocks, RT_HIST_THREADS, smem, stream>>>(pts, n, g, width, bins, hist, use_smem);
  return cudaGetLastError();
}

cudaError_t launch_route_mask(const float4* pts, uint32_t n, const RouteGrid& g, const RouteSplit& sp, unsigned short* mask,
                              cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const uint32_t blocks = std::min<uint32_t>((n + RT_THREADS - 1) / RT_THREADS, 148u * 8u);
  k_route_mask<<<blocks, RT_THREADS, 0, stream>>>(pts, n, g, sp, mask);
  return cudaGetLastError();
}

}  // namespace cm
