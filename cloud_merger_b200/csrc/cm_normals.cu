// cm_normals.cu -- pcl::NormalEstimation with a radius search on the sorted cell keys for sm_100a.
//
// PCL 1.8.1 (features/impl/normal_3d.hpp, KdTreeFLANN, setRadiusSearch): for every finite query the finite points p with
// fl((dx*dx + dy*dy) + dz*dz) < r2 = (float)(radius * radius) -- the radius outlier removal's rule -- in FLANN's order,
// ascending (squared distance, index); then computeMeanAndCovarianceMatrix (nine float running sums in that order),
// pcl::eigen33, the curvature and flipNormalTowardsViewpoint. The per-neighbourhood arithmetic lives in cm_ne_math.h,
// shared with the C++ statement of the tests. Here:
//  * the cloud goes through the radius outlier removal's front end with cell edge radius * (1 + 2^-8) (keys + onesweep
//    sort + cell table) and the statistical removal's sorted-order gather;
//  * k_ne_warp: one warp per query, in sorted order. It walks the nine row segments of cm_cells.cuh 32 candidates at a time
//    and ballot-compacts the hits as keys (bits(d2) << 32) | input index -- for non-negative floats the integer order of
//    that key is exactly FLANN's (distance, index) order -- into a list of CM_NE_WARP_CAP keys in shared memory, sorts the
//    list (bitonic), runs the nine running sums (lanes 0..8, each a serial chain in list order: reassociating them would
//    change the bits) and lane 0 solves. A query whose list overflows goes to a queue;
//  * k_ne_cta: one CTA per queued query, a buffer of NE_CTA_BUF keys. Up to CM_NE_CTA_CAP neighbours one walk collects the
//    whole list. Beyond that the walk keeps the smallest keys: whenever the buffer holds more than CM_NE_CTA_CAP keys it is
//    sorted and cut to its NE_CTA_KEEP smallest, and from then on only keys up to the last kept one are taken. The end of
//    the walk leaves exactly the keys in (lower, bound], which feed the sums in order; the next walk starts above bound.
//    So a neighbourhood of any size -- up to the whole cloud -- is summed in FLANN's order with no memory beyond the
//    CTA's shared buffer, at the price of one walk per ~NE_CTA_KEEP neighbours.
// Both kernels are launched every call (the CTA grid exits at once on an empty queue): the launch plan does not depend on
// the data and nothing waits for the host.
#include "../../include/cloud_merger_gpu.h"  // CM_NE_WARP_CAP, CM_NE_CTA_CAP
#include "cm_cells.cuh"
#include "cm_ne_math.h"

namespace cm {

namespace {

constexpr int NE_WARPS = 8;
constexpr uint32_t NE_WARP_CAP = CM_NE_WARP_CAP;
constexpr int NE_CTA_THREADS = 256;
constexpr uint32_t NE_CTA_BUF = 8192;                       // keys of the CTA buffer (64 KB, a power of two)
constexpr uint32_t NE_CTA_CAP = NE_CTA_BUF - NE_CTA_THREADS;  // a chunk of candidates always fits behind it
constexpr uint32_t NE_CTA_KEEP = 4096;                      // keys kept when the buffer is cut
constexpr uint32_t NE_CTA_GRID = 1024;
constexpr uint32_t FULL = 0xFFFFFFFFu;
constexpr unsigned long long NO_KEY = ~0ull;
static_assert(NE_CTA_CAP == CM_NE_CTA_CAP, "CM_NE_CTA_CAP");

// FLANN's float squared distance of candidate j to the query, as a list key; NO_KEY when it is not below r2
__device__ __forceinline__ unsigned long long hit_key(const float4& q, const float4& d, float r2, uint32_t idx) {
  const float acc = flann_d2(q, d);
  return acc < r2 ? ((unsigned long long)__float_as_uint(acc) << 32) | idx : NO_KEY;
}

// ascending bitonic sort of a[0 .. n) (padded with NO_KEY to the next power of two, which must fit) by `threads` threads
// of index t; sync() is the barrier of those threads
template <typename Sync>
__device__ __forceinline__ void bitonic(unsigned long long* a, uint32_t n, uint32_t t, uint32_t threads, Sync sync) {
  uint32_t P = 1;
  while (P < n) P <<= 1;
  for (uint32_t e = n + t; e < P; e += threads) a[e] = NO_KEY;
  sync();
  for (uint32_t k = 2; k <= P; k <<= 1)
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t e = t; e < P; e += threads) {
        const uint32_t o = e ^ j;
        if (o > e) {
          const unsigned long long x = a[e], y = a[o];
          if ((x > y) == ((e & k) == 0)) { a[e] = y; a[o] = x; }
        }
      }
      sync();
    }
}

// the nine running sums over list[0 .. n) in list order, one whole warp: lane c < 9 adds term c of every neighbour
__device__ __forceinline__ void chains(const unsigned long long* list, uint32_t n, const float4* __restrict__ pts,
                                       uint32_t lane, float& acc) {
  for (uint32_t b = 0; b < n; b += 32) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (b + lane < n) v = __ldg(pts + (uint32_t)list[b + lane]);
    const uint32_t m = min(32u, n - b);
    for (uint32_t t = 0; t < m; ++t) {
      const float x = __shfl_sync(FULL, v.x, t), y = __shfl_sync(FULL, v.y, t), z = __shfl_sync(FULL, v.z, t);
      if (lane < 9) acc = __fadd_rn(acc, cm_ne::sum_term((int)lane, x, y, z));
    }
  }
}

__device__ __forceinline__ uint32_t cloud_of(const NeParams& e, uint32_t idx) {
  uint32_t c = 0;
  while (idx >= e.begin[c + 1]) ++c;
  return c;
}

// lane 0 of a warp whose lanes 0..8 hold the sums of n neighbours: the normal of query `me`; true when it is NaN
__device__ __forceinline__ bool solve_and_store(const NeParams& e, float acc, uint32_t n, uint32_t me, const float4& q,
                                                uint32_t lane) {
  float sums[9];
#pragma unroll
  for (int c = 0; c < 9; ++c) sums[c] = __shfl_sync(FULL, acc, c);
  if (lane != 0) return false;
  float out[4];
  if (n < 3) {
    for (int k = 0; k < 4; ++k) out[k] = __uint_as_float(cm_ne::QNAN_BITS);
  } else {
    const float p[3] = {q.x, q.y, q.z};
    cm_ne::solve<false>(sums, n, p, e.vp, out);
  }
  e.out[me] = make_float4(out[0], out[1], out[2], out[3]);
  return cm_ne::is_nan(out[0]);
}

template <typename KeyT, bool TABLE>
__global__ void __launch_bounds__(NE_WARPS * 32) k_ne_warp(const VoxelParams p, const NeParams e) {
  __shared__ unsigned long long s_list[NE_WARPS][NE_WARP_CAP];
  __shared__ uint32_t s_nan[CM_MAX_ZONES], s_max, s_warp;
  const uint32_t tid = threadIdx.x, w = tid >> 5, lane = tid & 31u;
  if (tid < CM_MAX_ZONES) s_nan[tid] = 0;
  if (tid == 0) { s_max = 0; s_warp = 0; }
  __syncthreads();
  const uint32_t M = p.frame_surv_start[p.n_frames];
  const uint32_t i = blockIdx.x * NE_WARPS + w;
  if (i < M) do {
    const Sorted<KeyT> s = sorted_of<KeyT>(p);
    const uint32_t me = s.val(i);
    if (i == 0 && lane == 0) check_cell_margin(p);
    QueryCell qc;
    bool skip;
    if (!query_cell<KeyT>(p, s, i, qc, skip)) {  // a non-finite query
      if (lane == 0) {
        const float nan = __uint_as_float(cm_ne::QNAN_BITS);
        e.out[me] = make_float4(nan, nan, nan, nan);
        atomicAdd(&s_nan[cloud_of(e, me)], 1u);
      }
      break;
    }
    if (skip) break;
    const float4 q = e.sorted_pts[i];
    unsigned long long* list = s_list[w];
    uint32_t n = 0;
    for (int rr = 0; rr < 9 && n <= NE_WARP_CAP; ++rr) {
      uint32_t lo, hi;
      unsigned long long k_hi;
      if (!row_segment<KeyT, TABLE>(s, e.cell_start, M, qc, rr, lo, hi, k_hi)) continue;
      for (uint32_t b = lo; b < hi && n <= NE_WARP_CAP; b += 32) {
        const uint32_t j = b + lane;
        bool in = j < hi;
        if (!TABLE && in) in = s.key(j) <= k_hi;
        const unsigned long long k = in ? hit_key(q, e.sorted_pts[j], e.r2, s.val(j)) : NO_KEY;
        const uint32_t hits = __ballot_sync(FULL, k != NO_KEY);
        const uint32_t pos = n + __popc(hits & ((1u << lane) - 1u));
        if (k != NO_KEY && pos < NE_WARP_CAP) list[pos] = k;
        n += __popc(hits);
        if (!TABLE && __any_sync(FULL, !in)) break;
      }
    }
    if (n > NE_WARP_CAP) {  // to the CTA path
      if (lane == 0) e.queue[atomicAdd(&e.stats->n_queue, 1u)] = i;
      break;
    }
    __syncwarp();
    bitonic(list, n, lane, 32u, []() { __syncwarp(); });
    float acc = 0.0f;
    chains(list, n, e.pts, lane, acc);
    if (solve_and_store(e, acc, n, me, q, lane)) atomicAdd(&s_nan[cloud_of(e, me)], 1u);
    if (lane == 0) { atomicMax(&s_max, n); atomicAdd(&s_warp, 1u); }
  } while (false);
  __syncthreads();
  if (tid < CM_MAX_ZONES && s_nan[tid]) atomicAdd(&e.stats->n_nan[tid], s_nan[tid]);
  if (tid == 0) {
    if (s_max) atomicMax(&e.stats->max_neighbors, s_max);
    if (s_warp) atomicAdd(&e.stats->n_warp, s_warp);
  }
}

template <typename KeyT, bool TABLE>
__global__ void __launch_bounds__(NE_CTA_THREADS) k_ne_cta(const VoxelParams p, const NeParams e) {
  extern __shared__ unsigned long long s_buf[];
  __shared__ uint32_t s_n, s_part[NE_CTA_THREADS / 32];
  __shared__ unsigned long long s_bound;
  const uint32_t tid = threadIdx.x, w = tid >> 5, lane = tid & 31u;
  const uint32_t M = p.frame_surv_start[p.n_frames];
  const uint32_t n_queue = e.stats->n_queue;
  const Sorted<KeyT> s = sorted_of<KeyT>(p);
  auto sync = []() { __syncthreads(); };
  for (uint32_t qi = blockIdx.x; qi < n_queue; qi += gridDim.x) {
    const uint32_t i = e.queue[qi];
    const uint32_t me = s.val(i);
    QueryCell qc;
    bool skip;
    query_cell<KeyT>(p, s, i, qc, skip);  // queued queries are finite and keyed
    const float4 q = e.sorted_pts[i];
    float acc = 0.0f;
    uint32_t total = 0, passes = 0;
    unsigned long long lower = 0;
    bool has_lower = false;
    for (;;) {  // one walk over the candidates per pass
      if (tid == 0) { s_n = 0; s_bound = NO_KEY; }
      __syncthreads();
      for (int rr = 0; rr < 9; ++rr) {
        uint32_t lo, hi;
        unsigned long long k_hi;
        if (!row_segment<KeyT, TABLE>(s, e.cell_start, M, qc, rr, lo, hi, k_hi)) continue;
        for (uint32_t b = lo; b < hi; b += NE_CTA_THREADS) {
          const uint32_t j = b + tid;
          bool in = j < hi;
          if (!TABLE && in) in = s.key(j) <= k_hi;
          unsigned long long k = in ? hit_key(q, e.sorted_pts[j], e.r2, s.val(j)) : NO_KEY;
          if (k != NO_KEY && ((has_lower && k <= lower) || k > s_bound)) k = NO_KEY;
          const uint32_t hits = __ballot_sync(FULL, k != NO_KEY);
          if (lane == 0) s_part[w] = hits ? atomicAdd(&s_n, (uint32_t)__popc(hits)) : 0u;
          __syncwarp();
          if (k != NO_KEY) s_buf[s_part[w] + __popc(hits & ((1u << lane) - 1u))] = k;
          const bool last = TABLE ? b + NE_CTA_THREADS >= hi : __syncthreads_or(!in) != 0;
          __syncthreads();
          if (s_n > NE_CTA_CAP) {  // cut the buffer to its NE_CTA_KEEP smallest keys
            bitonic(s_buf, s_n, tid, NE_CTA_THREADS, sync);
            if (tid == 0) { s_bound = s_buf[NE_CTA_KEEP - 1]; s_n = NE_CTA_KEEP; }
            __syncthreads();
          }
          if (last) break;
        }
      }
      const uint32_t n = s_n;
      bitonic(s_buf, n, tid, NE_CTA_THREADS, sync);
      if (w == 0) chains(s_buf, n, e.pts, lane, acc);
      total += n;
      ++passes;
      const unsigned long long bound = s_bound;
      __syncthreads();
      if (bound == NO_KEY) break;
      lower = bound;
      has_lower = true;
    }
    if (w == 0) {
      const bool is_nan = solve_and_store(e, acc, total, me, q, lane);
      if (lane == 0) {
        if (is_nan) atomicAdd(&e.stats->n_nan[cloud_of(e, me)], 1u);
        atomicMax(&e.stats->max_neighbors, total);
        atomicAdd(passes == 1 ? &e.stats->n_cta : &e.stats->n_multi, 1u);
      }
    }
    __syncthreads();
  }
}

}  // namespace

cudaError_t configure_normal_kernels() {
  const int bytes = (int)(NE_CTA_BUF * sizeof(unsigned long long));
  cudaError_t err = cudaSuccess;
  auto set = [&](const void* f) {
    if (err == cudaSuccess) err = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  };
  set((const void*)k_ne_cta<uint32_t, true>);
  set((const void*)k_ne_cta<uint32_t, false>);
  set((const void*)k_ne_cta<unsigned long long, true>);
  set((const void*)k_ne_cta<unsigned long long, false>);
  return err;
}

int launch_normals(const VoxelParams& p, const NeParams& e, float4* sorted_pts, cudaStream_t stream, cudaEvent_t mid,
                   cudaError_t* err) {
  *err = cudaSuccess;
  if (p.max_points == 0) return 0;
  *err = launch_sorted_gather(p, sorted_pts, stream);
  if (*err != cudaSuccess) return 0;
  const uint32_t wb = (p.max_points + NE_WARPS - 1) / NE_WARPS;
  const uint32_t cb = std::min<uint32_t>(p.max_points, NE_CTA_GRID);
  const size_t smem = NE_CTA_BUF * sizeof(unsigned long long);
  with_cells(p, e.cell_start, [&](auto key, auto table) {
    using KeyT = decltype(key);
    constexpr bool TABLE = decltype(table)::value;
    k_ne_warp<KeyT, TABLE><<<wb, NE_WARPS * 32, 0, stream>>>(p, e);
    if (mid) cudaEventRecord(mid, stream);
    k_ne_cta<KeyT, TABLE><<<cb, NE_CTA_THREADS, smem, stream>>>(p, e);
  });
  *err = cudaGetLastError();
  return 3;
}

}  // namespace cm
