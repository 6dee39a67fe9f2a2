// cm_statistical.cu -- pcl::StatisticalOutlierRemoval on the sorted cell keys for sm_100a.
//
// PCL 1.8.1 (filters/impl/statistical_outlier_removal.hpp, applyFilterIndices): for every finite point the mean_k + 1
// nearest squared distances of an exact FLANN search (the point itself first, float squared distances in L2_Simple's order
// (dx*dx + dy*dy) + dz*dz), dist_sum += sqrt(nn_dists[k]) over k = 1 .. mean_k in ascending order (a double), the point's
// distance (float)(dist_sum / mean_k); 0 for a non-finite point. Then double sums of the distances and of their float
// squares over the cloud in index order, mean, stddev and threshold = mean + std_mul * stddev, and a point is removed iff
// its distance > threshold (negative: <=).
//
// Here the cloud goes through the VoxelGrid front end with a cell edge chosen by the host (keys + onesweep sort, as the
// radius outlier removal does), the points are gathered into sorted order, and one warp per point finds the exact
// mean_k + 1 smallest float squared distances by visiting growing cubes of cells around its own (k_sor_knn):
//  * the running set lives in registers, slot s = j * 32 + lane (up to 4 per lane); candidates are scored 32 at a time,
//    a ballot against the current largest kept value filters them, and survivors replace that value one by one;
//  * the cube grows from half-width 0 by max(1, r / 2) at a time; a grown cube is visited as the row segments (x runs of
//    one (z, y) row of cells: one contiguous range of the sorted keys) that the previous cube did not cover;
//  * the search stops once every point outside the cube provably has a float squared distance >= the largest kept value
//    (the bound, DESIGN section 8, covers the float rounding of floor(x * inv) at any coordinate magnitude);
//  * the kept values are ranked in the warp and lane 0 adds their roots in ascending order, as PCL's loop does.
// k_sor_sums (one CTA per cloud) forms both double sums bit-exactly: in parallel when every value is a multiple of 2^e_min
// and the total stays below 2^(53 + e_min) -- then no partial sum of any order rounds -- and as the serial chain in index
// order otherwise. k_sor_select then sets the zone-slicing mask bit of every kept point (zone = cloud), and the zone
// scan + scatter kernels compact the survivors in input order (cm_zones.cu).
#include <climits>

#include "cm_cells.cuh"

namespace cm {

namespace {

constexpr int SOR_WARPS = 8;
constexpr int SOR_THREADS = SOR_WARPS * 32;
constexpr int SUM_THREADS = 1024;
constexpr int SERIAL_TILE = 4096;
constexpr uint32_t FULL = 0xFFFFFFFFu;

template <typename KeyT>
__global__ void __launch_bounds__(256) k_sor_gather(const VoxelParams p, float4* __restrict__ sorted_pts) {
  const uint32_t M = p.frame_surv_start[p.n_frames];
  const uint32_t i = blockIdx.x * 256 + threadIdx.x;
  if (i >= M) return;
  sorted_pts[i] = __ldg(p.pts + sorted_of<KeyT>(p).val(i));
}

// largest kept value and its slot (j * 32 + lane), the same in every lane; ties go to the lowest slot
template <int NS>
__device__ __forceinline__ float warp_argmax(const float (&v)[NS], uint32_t lane, uint32_t& own) {
  float m = v[0];
  uint32_t code = lane;
#pragma unroll
  for (int j = 1; j < NS; ++j)
    if (v[j] > m) { m = v[j]; code = (uint32_t)j * 32u + lane; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(FULL, m, o);
    const uint32_t oc = __shfl_xor_sync(FULL, code, o);
    if (om > m || (om == m && oc < code)) { m = om; code = oc; }
  }
  own = code;
  return m;
}

template <typename KeyT, bool TABLE, int NS>
__global__ void __launch_bounds__(SOR_THREADS, 2) k_sor_knn(const VoxelParams p, const SorParams s) {
  __shared__ float s_val[SOR_WARPS][32 * NS];
  __shared__ double s_root[SOR_WARPS][32 * NS];
  const uint32_t wib = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const uint32_t M = p.frame_surv_start[p.n_frames];
  const uint32_t i = blockIdx.x * SOR_WARPS + wib;  // one warp per sorted position
  if (i >= M) return;
  const Sorted<KeyT> st = sorted_of<KeyT>(p);
  const uint32_t idx_bits = p.info->idx_bits;
  const unsigned long long full_key = st.key(i);
  // clouds are frames of the key; keys of frame >= n_frames are the non-finite points (distance 0: the caller cleared it)
  const unsigned long long frame = idx_bits >= 64 ? 0ull : (full_key >> idx_bits);
  if (frame >= p.n_frames || ((s.too_few >> frame) & 1u)) return;
  const unsigned long long fbits = idx_bits >= 64 ? 0ull : (frame << idx_bits);
  const GridDev g = p.grid[frame];
  if (g.zero_keys) return;  // the host refuses such a call before this kernel is enqueued
  // query_cell's decode, in signed arithmetic for the cube bounds (on query_cell one instantiation takes two more
  // registers, DESIGN section 4)
  const long long d0 = g.div_b[0], d1 = g.div_b[1], d2 = g.div_b[2];
  const unsigned long long key = full_key - fbits;
  const long long c0 = (long long)(key % (unsigned long long)d0), t = (long long)(key / (unsigned long long)d0);
  const long long c1 = t % d1, c2 = t / d1;
  const float4 q = s.sorted_pts[i];
  // eps: how far (in cells) the float product x * inv of a point of this frame may lie from the exact one, twice -- every
  // |x * inv| of the frame is below max(|min_b|, |max_b|) + 1, and round-to-nearest errs by at most 2^-24 of it
  int mb = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) mb = max(mb, max(abs(g.min_b[a]), abs(g.max_b[a])));
  const double eps = ((double)mb + 1.0) * 0x1p-23 * (1.0 + 0x1p-20) + 0x1p-140;
  const uint32_t kp1 = s.mean_k + 1u;
  float v[NS];
#pragma unroll
  for (int j = 0; j < NS; ++j) v[j] = (uint32_t)j * 32u + lane < kp1 ? __int_as_float(0x7F800000) : -1.0f;
  float* buf = s_val[wib];
  uint32_t filled = 0, own = 0;
  float thr = __int_as_float(0x7F800000);
  long long r_old = -1, r = 0;
  while (true) {
    const long long zl = max(c2 - r, 0ll), zh = min(c2 + r, d2 - 1), yl = max(c1 - r, 0ll), yh = min(c1 + r, d1 - 1);
    const long long xl = max(c0 - r, 0ll), xh = min(c0 + r, d0 - 1);
    const long long ny = yh - yl + 1, pieces = 2 * (zh - zl + 1) * ny;
    // piece 2 row + side: a row of the cube outside the previous one is one segment (side 0); a row through the previous
    // cube leaves a segment on each side of it
    for (long long base = 0; base < pieces; base += 32) {
      const long long tp = base + lane;
      uint32_t lo = 0, cnt = 0;
      if (tp < pieces) {
        const long long row = tp >> 1, zz = zl + row / ny, yy = yl + row % ny;
        const bool side = (tp & 1) != 0;
        long long a = xl, b = xh;
        const bool outer = r_old < 0 || llabs(zz - c2) > r_old || llabs(yy - c1) > r_old;
        if (outer) { if (side) b = a - 1; }
        else if (!side) b = min(b, c0 - r_old - 1);
        else a = max(a, c0 + r_old + 1);
        if (a <= b) {
          const unsigned long long rowk = fbits + (unsigned long long)((zz * d1 + yy) * d0);
          uint32_t hi;
          if constexpr (TABLE) {
            lo = __ldg(s.cell_start + rowk + a);
            hi = __ldg(s.cell_start + rowk + b + 1);
          } else {
            lo = lower_bound(st, M, rowk + a);
            hi = lower_bound(st, M, rowk + b + 1);
          }
          cnt = hi - lo;
        }
      }
      // the lanes' segments, end to end: candidate j lies in the segment of the first lane whose inclusive sum exceeds j
      const uint32_t incl = warp_incl_scan_u32(cnt);
      const uint32_t total = __shfl_sync(FULL, incl, 31);
      for (uint32_t cb = 0; cb < total; cb += 32) {
        const uint32_t j = cb + lane;
        uint32_t L = 0;
#pragma unroll
        for (uint32_t step = 16; step; step >>= 1)
          if (__shfl_sync(FULL, incl, L + step - 1) <= j) L += step;
        const uint32_t seg_lo = __shfl_sync(FULL, lo, L), seg_ex = __shfl_sync(FULL, incl - cnt, L);
        const bool valid = j < total;
        float d = 0.f;
        if (valid) {
          d = flann_d2(q, s.sorted_pts[seg_lo + (j - seg_ex)]);
        }
        const bool filling = filled < kp1;
        const bool take = valid && (filling || d < thr);
        const uint32_t bal = __ballot_sync(FULL, take);
        if (!bal) continue;
        const uint32_t n_take = __popc(bal);
        if (take) buf[__popc(bal & lanemask_lt())] = d;
        __syncwarp();
        uint32_t first = 0;
        if (filling) {  // free slots are taken in order
          first = min(n_take, kp1 - filled);
#pragma unroll
          for (int jj = 0; jj < NS; ++jj) {
            const uint32_t sl = (uint32_t)jj * 32u + lane;
            if (sl >= filled && sl < filled + first) v[jj] = buf[sl - filled];
          }
          filled += first;
          if (filled == kp1) thr = warp_argmax<NS>(v, lane, own);
        }
        for (uint32_t k = first; k < n_take; ++k) {  // the rest replace the largest kept value
          const float dk = buf[k];
          if (!(dk < thr)) continue;
#pragma unroll
          for (int jj = 0; jj < NS; ++jj)
            if ((uint32_t)jj * 32u + lane == own) v[jj] = dk;
          thr = warp_argmax<NS>(v, lane, own);
        }
        __syncwarp();
      }
    }
    if (xl == 0 && xh == d0 - 1 && yl == 0 && yh == d1 - 1 && zl == 0 && zh == d2 - 1) break;  // the whole grid
    if (filled == kp1) {
      if (thr <= 0.f) break;
      // every point outside the cube is at least (r - eps) cells away on some axis; its float squared distance is then
      // >= ((r - eps) h)^2 (1 - 2^-24)^3 with h = 1 / inv (DESIGN section 8)
      const double m = (double)r - eps;
      if (m > 0.0) {
        const double a = m * s.cell;
        const double bound = a * a * (1.0 - 0x1p-20);
        if (bound >= 0x1p-100 && bound >= (double)thr) break;
      }
    }
    r_old = r;
    r += max(1ll, r >> 1);
  }
  // ascending order: rank every kept value (ties by slot), then lane 0 adds the roots as PCL's loop does
#pragma unroll
  for (int j = 0; j < NS; ++j) {
    const uint32_t sl = (uint32_t)j * 32u + lane;
    if (sl < kp1) buf[sl] = v[j];
  }
  __syncwarp();
  double* root = s_root[wib];
#pragma unroll
  for (int j = 0; j < NS; ++j) {
    const uint32_t sl = (uint32_t)j * 32u + lane;
    if (sl >= kp1) continue;
    uint32_t rank = 0;
    for (uint32_t u = 0; u < kp1; ++u) {
      const float w = buf[u];
      rank += (w < v[j] || (w == v[j] && u < sl)) ? 1u : 0u;
    }
    root[rank] = s.sqrt_mode ? __dsqrt_rn((double)v[j]) : (double)__fsqrt_rn(v[j]);
  }
  __syncwarp();
  if (lane == 0) {
    double sum = 0.0;
    for (uint32_t k = 1; k < kp1; ++k) sum = __dadd_rn(sum, root[k]);  // k = 0 is the point itself
    s.dist[st.val(i)] = __double2float_rn(__ddiv_rn(sum, (double)s.mean_k));
  }
}

// exponent of the lowest set bit of a non-negative float (INT_MAX for 0)
__device__ __forceinline__ int lsb_exp(float v) {
  const uint32_t b = __float_as_uint(v) & 0x7FFFFFFFu;
  if (!b) return INT_MAX;
  const uint32_t ex = b >> 23, man = b & 0x7FFFFFu;
  return ex ? (int)ex - 150 + (__ffs(man | 0x800000u) - 1) : -149 + (__ffs(man) - 1);
}

__global__ void __launch_bounds__(SUM_THREADS) k_sor_sums(const SorSumParams s) {
  const uint32_t c = blockIdx.x, tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
  const uint32_t b = s.begin[c], e = s.begin[c + 1];
  __shared__ double s_tot[2][32];
  __shared__ int s_emin[2][32];
  __shared__ uint32_t s_bad[32];
  __shared__ float s_tile[SERIAL_TILE];
  __shared__ uint32_t s_serial;
  // any-order double totals, the lowest set bit of every value, non-finite values
  double ts = 0.0, tq = 0.0;
  int es = INT_MAX, eq = INT_MAX;
  uint32_t bad = 0;
  for (uint32_t i = b + tid; i < e; i += SUM_THREADS) {
    const float v = s.dist[i], v2 = __fmul_rn(v, v);
    ts = __dadd_rn(ts, (double)v);
    tq = __dadd_rn(tq, (double)v2);
    es = min(es, lsb_exp(v));
    eq = min(eq, lsb_exp(v2));
    if (!finite_f32(v) || v < 0.f) bad |= 1u;
    if (!finite_f32(v2)) bad |= 2u;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ts = __dadd_rn(ts, __shfl_xor_sync(FULL, ts, o));
    tq = __dadd_rn(tq, __shfl_xor_sync(FULL, tq, o));
    es = min(es, __shfl_xor_sync(FULL, es, o));
    eq = min(eq, __shfl_xor_sync(FULL, eq, o));
    bad |= __shfl_xor_sync(FULL, bad, o);
  }
  if (lane == 0) { s_tot[0][w] = ts; s_tot[1][w] = tq; s_emin[0][w] = es; s_emin[1][w] = eq; s_bad[w] = bad; }
  __syncthreads();
  if (tid == 0) {
    for (int k = 1; k < SUM_THREADS / 32; ++k) {
      ts = __dadd_rn(ts, s_tot[0][k]); tq = __dadd_rn(tq, s_tot[1][k]);
      es = min(es, s_emin[0][k]); eq = min(eq, s_emin[1][k]); bad |= s_bad[k];
    }
    // With non-negative values every partial sum of any order is at most the exact total; below 2^(53 + e_min) all of
    // them are exact multiples of 2^e_min, so the order does not matter. The computed total reaches 2^(53 + e_min) iff
    // the exact one does (round-to-nearest is monotone and the bound is a double), so the test needs no exact total.
    uint32_t serial = s.force_serial ? 3u : 0u;
    if ((bad & 1u) || (es != INT_MAX && !(ts < ldexp(1.0, 53 + es)))) serial |= 1u;
    if ((bad & 2u) || (eq != INT_MAX && !(tq < ldexp(1.0, 53 + eq)))) serial |= 2u;
    s_serial = serial;
    s_tot[0][0] = ts; s_tot[1][0] = tq;
  }
  __syncthreads();
  const uint32_t serial = s_serial;
  double sum = s_tot[0][0], sq_sum = s_tot[1][0];
  if (serial) {  // PCL's loop: sum += d, sq_sum += d * d (a float product), index order
    double cs = 0.0, cq = 0.0;
    for (uint32_t t0 = b; t0 < e; t0 += SERIAL_TILE) {
      const uint32_t n = min((uint32_t)SERIAL_TILE, e - t0);
      for (uint32_t k = tid; k < n; k += SUM_THREADS) s_tile[k] = s.dist[t0 + k];
      __syncthreads();
      if (tid == 0) {
        if (serial == 3u) {
          for (uint32_t k = 0; k < n; ++k) {
            const float v = s_tile[k];
            cs = __dadd_rn(cs, (double)v);
            cq = __dadd_rn(cq, (double)__fmul_rn(v, v));
          }
        } else if (serial == 1u) {
          for (uint32_t k = 0; k < n; ++k) cs = __dadd_rn(cs, (double)s_tile[k]);
        } else {
          for (uint32_t k = 0; k < n; ++k) cq = __dadd_rn(cq, (double)__fmul_rn(s_tile[k], s_tile[k]));
        }
      }
      __syncthreads();
    }
    if (serial & 1u) sum = cs;
    if (serial & 2u) sq_sum = cq;
  }
  if (tid == 0) {
    const double valid = (double)s.n_valid[c];
    SorStats st;
    st.sum = sum;
    st.sq_sum = sq_sum;
    st.mean = __ddiv_rn(sum, valid);
    const double variance = __ddiv_rn(__dsub_rn(sq_sum, __ddiv_rn(__dmul_rn(sum, sum), valid)), __dsub_rn(valid, 1.0));
    st.stddev = __dsqrt_rn(variance);
    st.threshold = __dadd_rn(st.mean, __dmul_rn(s.std_mul, st.stddev));
    st.path = serial;
    st.pad_ = 0;
    s.stats[c] = st;
  }
}

__global__ void __launch_bounds__(256) k_sor_select(const SorSumParams s, uint32_t n) {
  const uint32_t i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  uint32_t c = 0;
  while (i >= s.begin[c + 1]) ++c;
  const double d = (double)s.dist[i], thr = s.stats[c].threshold;
  // a NaN threshold keeps every point either way, as in PCL
  const bool removed = ((s.too_few >> c) & 1u) ? false : (s.negative ? d <= thr : d > thr);
  s.mask[i] = removed ? (unsigned short)0 : (unsigned short)(1u << c);  // zone = cloud
}

}  // namespace

cudaError_t launch_sorted_gather(const VoxelParams& p, float4* sorted_pts, cudaStream_t stream) {
  if (p.max_points == 0) return cudaSuccess;
  const uint32_t gb = (p.max_points + 255) / 256;
  with_key_type(p, [&](auto key) { k_sor_gather<decltype(key)><<<gb, 256, 0, stream>>>(p, sorted_pts); });
  return cudaGetLastError();
}

cudaError_t launch_sor_knn(const VoxelParams& p, const SorParams& s, float4* sorted_pts, cudaStream_t stream) {
  if (p.max_points == 0) return cudaSuccess;
  const cudaError_t ge = launch_sorted_gather(p, sorted_pts, stream);
  if (ge != cudaSuccess) return ge;
  const uint32_t blocks = (p.max_points + SOR_WARPS - 1) / SOR_WARPS;
  const int ns = s.mean_k + 1 <= 32 ? 1 : s.mean_k + 1 <= 64 ? 2 : 4;
  with_cells(p, s.cell_start, [&](auto key, auto table) {
    using KeyT = decltype(key);
    constexpr bool TABLE = decltype(table)::value;
    if (ns == 1) k_sor_knn<KeyT, TABLE, 1><<<blocks, SOR_THREADS, 0, stream>>>(p, s);
    else if (ns == 2) k_sor_knn<KeyT, TABLE, 2><<<blocks, SOR_THREADS, 0, stream>>>(p, s);
    else k_sor_knn<KeyT, TABLE, 4><<<blocks, SOR_THREADS, 0, stream>>>(p, s);
  });
  return cudaGetLastError();
}

cudaError_t launch_sor_sums(const SorSumParams& s, cudaStream_t stream) {
  k_sor_sums<<<s.n_clouds, SUM_THREADS, 0, stream>>>(s);
  return cudaGetLastError();
}

cudaError_t launch_sor_select(const SorSumParams& s, uint32_t n_points, cudaStream_t stream) {
  if (n_points == 0) return cudaSuccess;
  k_sor_select<<<(n_points + 255) / 256, 256, 0, stream>>>(s, n_points);
  return cudaGetLastError();
}

}  // namespace cm
