// cm_plane.cu -- RANSAC ground plane (pcl::SACSegmentation, SACMODEL_PLANE / PERPENDICULAR_PLANE / PARALLEL_PLANE +
// SAC_RANSAC) for sm_100a.
//
// Replaces the plane search of removeGround() in the reference (pcl_preprocessing/src/pc_preprocessing_main.cpp:95-117;
// parameters Parameter.h:38-42: 1000 iterations, threshold 0.3 m, probability 0.99, optimize on). PCL 1.8.1 evaluates one
// hypothesis after the other: draw three indices, fit the plane through them, count the points within the threshold, lower
// the iteration bound k from the best count so far, stop when iterations >= k. The three-index draws come from a
// fixed-seed Mersenne twister and do not depend on the data, so the host generates the draw stream ahead, and
//
//   k_plane_score   fits and scores a whole batch of draws at once, for up to eight independent clouds (blockIdx.z; the
//                   zones of one sensor cloud): blockIdx.y picks 128 draws (one per thread), blockIdx.x a chunk of
//                   512 points staged in shared memory and broadcast to the 128 threads; per draw the kernel
//                   writes the sample test (isSampleGood) and the axis test of the constrained models (isModelValid;
//                   a model that fails it skips the point loop: 0 inliers), the model and the inlier count. The host then walks the batch
//                   in draw order with PCL's stopping rule -- the result is the model PCL's sequential loop ends on.
//   k_plane_select  selectWithinDistance with the final model of every cloud: inlier / rest flags of every point (bits 2k /
//                   2k + 1 of the zone-slicing mask for cloud k; its scan + scatter kernels produce the ground and
//                   no-ground clouds in input order, as the two pcl::ExtractIndices passes of the reference do).
//   k_plane_moments optimizeModelCoefficients' running sums (xx, xy, xz, yy, yz, zz, x, y, z over the inliers of the RANSAC
//                   model) in PCL's order: float accumulators, one add per inlier in index order. Nine lanes of one warp
//                   carry the nine serial chains while eight producer warps test the next 256 points against the model,
//                   compact the inliers among them and stage their products (double buffer). One CTA per cloud.
//
// All float arithmetic is single IEEE operations in PCL's / Eigen's order (no FMA); the order of Eigen's 4-wide packet
// reductions depends on the instruction set PCL was built for and is a parameter (PlaneParams::sum_order).
//
// Roofline: k_plane_score is FP32-issue bound (8 instructions per point x draw) and takes ~12 us per batch; the serial sums
// of k_plane_moments are latency-bound by definition (5.9 cycles per inlier measured, 4 is the FADD latency) and are the
// kernel time of the call; the rest of its wall time is three host round trips (scores -> stopping rule, sums -> 3 x 3
// solve, final counts).
#include <algorithm>

#include "cm_kernels.h"

namespace cm {

namespace {

constexpr int PL_THREADS = 128;  // draws per CTA
constexpr int PL_CHUNK = 512;    // points per CTA

template <int ORDER>
__device__ __forceinline__ float sum4(float l0, float l1, float l2, float l3) {
  if constexpr (ORDER == 0) return __fadd_rn(__fadd_rn(l0, l2), __fadd_rn(l1, l3));
  else if constexpr (ORDER == 1) return __fadd_rn(__fadd_rn(l0, l1), __fadd_rn(l2, l3));
  else return __fadd_rn(__fadd_rn(__fadd_rn(l0, l1), l2), l3);
}

// Eigen 3.3 normalize(): only when the squared norm is positive
template <int ORDER>
__device__ __forceinline__ float4 normalized(float4 c) {
  const float z = sum4<ORDER>(__fmul_rn(c.x, c.x), __fmul_rn(c.y, c.y), __fmul_rn(c.z, c.z), __fmul_rn(c.w, c.w));
  if (z > 0.f) {
    const float nrm = __fsqrt_rn(z);
    c.x = __fdiv_rn(c.x, nrm); c.y = __fdiv_rn(c.y, nrm); c.z = __fdiv_rn(c.z, nrm); c.w = __fdiv_rn(c.w, nrm);
  }
  return c;
}

template <int ORDER>
__device__ __forceinline__ float plane_abs_dist(const float4 c, const float4 q) {
  return fabsf(sum4<ORDER>(__fmul_rn(c.x, q.x), __fmul_rn(c.y, q.y), __fmul_rn(c.z, q.z), c.w));
}

template <int ORDER>
__global__ void __launch_bounds__(PL_THREADS) k_plane_score(const PlaneParams p) {
  __shared__ float4 s_pts[PL_CHUNK];
  const uint32_t cloud = blockIdx.z;
  const uint32_t first = p.begin[cloud], n_here = p.begin[cloud + 1] - first, n_draws = p.n_draws[cloud];
  const uint32_t base = blockIdx.x * PL_CHUNK;
  if (base >= n_here || blockIdx.y * PL_THREADS >= n_draws) return;  // whole CTA: nothing of this cloud / batch here
  const float4* __restrict__ pts = p.pts + first;
  const float qnan = __int_as_float(0x7fc00000);
  for (int i = threadIdx.x; i < PL_CHUNK; i += PL_THREADS) {
    const uint32_t idx = base + i;
    s_pts[i] = idx < n_here ? __ldg(pts + idx) : make_float4(qnan, qnan, qnan, qnan);  // a NaN distance is never inside
  }
  const uint32_t h = blockIdx.y * PL_THREADS + threadIdx.x;
  const uint32_t slot = cloud * p.draw_stride + h;
  bool good = false, valid = true;
  float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
  if (h < n_draws) {
    const int32_t* smp = p.samples + 3 * (size_t)slot;
    const float4 p0 = __ldg(pts + smp[0]), p1 = __ldg(pts + smp[1]), p2 = __ldg(pts + smp[2]);
    const float ux = __fsub_rn(p1.x, p0.x), uy = __fsub_rn(p1.y, p0.y), uz = __fsub_rn(p1.z, p0.z);
    const float vx = __fsub_rn(p2.x, p0.x), vy = __fsub_rn(p2.y, p0.y), vz = __fsub_rn(p2.z, p0.z);
    // isSampleGood / the collinearity test of computeModelCoefficients: the quotients of the two edge vectors
    const float qx = __fdiv_rn(ux, vx), qy = __fdiv_rn(uy, vy), qz = __fdiv_rn(uz, vz);
    good = (qx != qy) || (qz != qy);
    c.x = __fsub_rn(__fmul_rn(uy, vz), __fmul_rn(uz, vy));
    c.y = __fsub_rn(__fmul_rn(uz, vx), __fmul_rn(ux, vz));
    c.z = __fsub_rn(__fmul_rn(ux, vy), __fmul_rn(uy, vx));
    c.w = 0.f;
    c = normalized<ORDER>(c);
    c.w = __fmul_rn(-1.0f, sum4<ORDER>(__fmul_rn(c.x, p0.x), __fmul_rn(c.y, p0.y), __fmul_rn(c.z, p0.z), __fmul_rn(c.w, 1.0f)));
    if (p.axis_rule.test) {
      // isModelValid of the axis-constrained models: (a, b, c, 0) normalized once more -- and a second time inside
      // getAngle3D for PERPENDICULAR -- dotted with the pre-normalized axis
      float4 m = normalized<ORDER>(make_float4(c.x, c.y, c.z, 0.f));
      if (p.axis_rule.test == 1) m = normalized<ORDER>(m);
      const float4 a = p.axis_rule.axis;
      const float d = sum4<ORDER>(__fmul_rn(a.x, m.x), __fmul_rn(a.y, m.y), __fmul_rn(a.z, m.z), __fmul_rn(a.w, m.w));
      valid = plane_axis_valid(p.axis_rule, d);
    }
    if (blockIdx.x == 0) {
      p.models[slot] = c;
      p.good[slot] = !good ? 0 : valid ? 1 : 2;
    }
  }
  __syncthreads();
  if (!good || !valid) return;  // an invalid model counts 0 inliers (countWithinDistance)
  int cnt = 0;
#pragma unroll 8
  for (int i = 0; i < PL_CHUNK; ++i) cnt += plane_abs_dist<ORDER>(c, s_pts[i]) < p.threshold ? 1 : 0;
  if (cnt) atomicAdd(p.counts + slot, cnt);
}

// inliers of cloud k -> bit 2k, its other points -> bit 2k + 1 (a cloud without a model: everything is "other")
template <int ORDER>
__global__ void __launch_bounds__(256) k_plane_select(const PlaneSelect q) {
  const uint32_t i = blockIdx.x * 256u + threadIdx.x;
  if (i >= q.begin[q.n_clouds]) return;
  uint32_t k = 0;
  while (i >= q.begin[k + 1]) ++k;
  const bool in = q.found[k] && plane_abs_dist<ORDER>(q.coeff[k], __ldg(q.pts + i)) < q.threshold;
  q.mask[i] = (unsigned short)((in ? 1u : 2u) << (2u * k));
}

// 16 staged terms as four 16-byte shared-memory loads
__device__ __forceinline__ void ld16_shared(float (&v)[16], const float* row) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const float4 x = *reinterpret_cast<const float4*>(row + 4 * u);
    v[4 * u] = x.x; v[4 * u + 1] = x.y; v[4 * u + 2] = x.z; v[4 * u + 3] = x.w;
  }
}
__device__ __forceinline__ void add16_chain(float& acc, const float (&v)[16]) {
#pragma unroll
  for (int u = 0; u < 16; ++u) acc = __fadd_rn(acc, v[u]);
}

constexpr int PM_TILE = 256;
constexpr int PM_WARPS = PM_TILE / 32;     // producer warps
constexpr int PM_STRIDE = PM_TILE + 20;  // 16-byte aligned rows; the adding warp prefetches up to 16 terms past a full tile
constexpr int PM_THREADS = 32 + PM_TILE;  // warp 0 accumulates, the others select and stage

// One CTA per cloud. Producer warps: test 256 points of the cloud against its RANSAC model (selectWithinDistance), compact
// the inliers of the tile in index order (ballot + warp counts) and stage their nine products; warp 0: nine lanes add the
// staged terms of the previous tile to the nine running sums, one add per inlier, in order.
template <int ORDER>
__global__ void __launch_bounds__(PM_THREADS) k_plane_moments(const PlaneSelect q,
                                                             float* __restrict__ out_all /* per cloud: [9] sums, [1] count bits */) {
  __shared__ __align__(16) float s_term[2][9][PM_STRIDE];  // rows 16-byte aligned: the chains read float4
  __shared__ int s_wcnt[2][PM_WARPS];
  __shared__ int s_cnt[2];
  const uint32_t cloud = blockIdx.x;
  const uint32_t first = q.begin[cloud], n = q.begin[cloud + 1] - first;
  float* __restrict__ out = out_all + 16 * cloud;
  if (!q.found[cloud] || n == 0) {
    if (threadIdx.x < 10) out[threadIdx.x] = 0.f;
    return;
  }
  const float4* __restrict__ pts = q.pts + first;
  const float4 c = q.coeff[cloud];
  const uint32_t n_tiles = (n + PM_TILE - 1) / PM_TILE;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j = (int)threadIdx.x - 32;  // producers: the point of the tile this thread tests
  float acc = 0.f;
  uint32_t n_in = 0;
#ifdef CM_PLANE_CYCLES
  const long long c_begin = clock64();
  long long c_busy = 0;
#endif
  const float qnan = __int_as_float(0x7fc00000);
  float4 pt = make_float4(qnan, qnan, qnan, qnan);
  if (warp > 0 && (uint32_t)j < n) pt = __ldg(pts + j);
  for (uint32_t t = 0; t <= n_tiles; ++t) {
    if (warp > 0) {
      if (t < n_tiles) {
        const uint32_t idx = t * PM_TILE + j;
        float4 pt_next = make_float4(qnan, qnan, qnan, qnan);
        if (idx + PM_TILE < n) pt_next = __ldg(pts + idx + PM_TILE);  // in flight across the barriers
        const bool in = plane_abs_dist<ORDER>(c, pt) < q.threshold;  // out-of-range lanes hold NaN: never inside
        const uint32_t bal = __ballot_sync(0xffffffffu, in);
        if (lane == 0) s_wcnt[t & 1][warp - 1] = __popc(bal);
        asm volatile("bar.sync 1, %0;" ::"n"(PM_TILE) : "memory");  // the producer warps only
        int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < PM_WARPS; ++w) {
          const int cw = s_wcnt[t & 1][w];
          before += w < warp - 1 ? cw : 0;
          total += cw;
        }
        if (in) {
          const int pos = before + __popc(bal & ((1u << lane) - 1u));
          float(*term)[PM_STRIDE] = s_term[t & 1];
          term[0][pos] = __fmul_rn(pt.x, pt.x);
          term[1][pos] = __fmul_rn(pt.x, pt.y);
          term[2][pos] = __fmul_rn(pt.x, pt.z);
          term[3][pos] = __fmul_rn(pt.y, pt.y);
          term[4][pos] = __fmul_rn(pt.y, pt.z);
          term[5][pos] = __fmul_rn(pt.z, pt.z);
          term[6][pos] = pt.x;
          term[7][pos] = pt.y;
          term[8][pos] = pt.z;
        }
        // pad the tile to whole pairs of 16-term groups with +0.0f (x + 0 == x for every running sum: it starts at +0
        // and can never become -0), so the adding warp runs a branch-free loop without a remainder
        const int pad = ((total + 31) & ~31) - total;
        if (j < pad) {
#pragma unroll
          for (int r = 0; r < 9; ++r) s_term[t & 1][r][total + j] = 0.f;
        }
        if (j == 0) s_cnt[t & 1] = total;
        pt = pt_next;
      }
    } else if (t > 0) {
      const int cnt = s_cnt[(t - 1) & 1];
      n_in += (uint32_t)cnt;
#ifdef CM_PLANE_CYCLES
      const long long c0 = clock64();
#endif
      if (lane < 9) {
        // the serial chain: two sets of 16 terms, the loads of one set in flight during the 16 dependent adds of the other.
        // No branch inside the loop body: ptxas waits for all outstanding loads at a branch, which would expose their
        // latency twice per iteration (measured: 7.6 instead of 4.3 cycles per add). The last prefetch reads past the
        // padded tile (inside the row's slack) and is never added.
        const float* row = s_term[(t - 1) & 1][lane];
        const int pairs = (cnt + 31) >> 5;
        float va[16], vb[16];
        ld16_shared(va, row);
#pragma unroll 1
        for (int pr = 0; pr < pairs; ++pr) {
          ld16_shared(vb, row + 32 * pr + 16);
          add16_chain(acc, va);
          ld16_shared(va, row + 32 * pr + 32);
          add16_chain(acc, vb);
        }
      }
#ifdef CM_PLANE_CYCLES
      c_busy += clock64() - c0;
#endif
    }
    __syncthreads();
  }
  if (warp == 0 && lane < 9) out[lane] = acc;
  if (threadIdx.x == 0) out[9] = __uint_as_float(n_in);
#ifdef CM_PLANE_CYCLES
  if (threadIdx.x == 0) {
    out[10] = __uint_as_float((uint32_t)(clock64() - c_begin));
    out[11] = __uint_as_float((uint32_t)c_busy);
  }
#endif
}

}  // namespace

cudaError_t launch_plane_score(const PlaneParams& p, cudaStream_t stream) {
  uint32_t max_points = 0, max_draws = 0;
  for (uint32_t k = 0; k < p.n_clouds; ++k) {
    if (!p.n_draws[k]) continue;
    max_points = std::max(max_points, p.begin[k + 1] - p.begin[k]);
    max_draws = std::max(max_draws, p.n_draws[k]);
  }
  if (max_points == 0 || max_draws == 0) return cudaSuccess;
  const dim3 grid((max_points + PL_CHUNK - 1) / PL_CHUNK, (max_draws + PL_THREADS - 1) / PL_THREADS, p.n_clouds);
  if (p.sum_order == 0) k_plane_score<0><<<grid, PL_THREADS, 0, stream>>>(p);
  else if (p.sum_order == 1) k_plane_score<1><<<grid, PL_THREADS, 0, stream>>>(p);
  else k_plane_score<2><<<grid, PL_THREADS, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_plane_select(const PlaneSelect& q, uint32_t sum_order, cudaStream_t stream) {
  const uint32_t n = q.begin[q.n_clouds];
  if (n == 0) return cudaSuccess;
  const uint32_t blocks = (n + 255u) / 256u;
  if (sum_order == 0) k_plane_select<0><<<blocks, 256, 0, stream>>>(q);
  else if (sum_order == 1) k_plane_select<1><<<blocks, 256, 0, stream>>>(q);
  else k_plane_select<2><<<blocks, 256, 0, stream>>>(q);
  return cudaGetLastError();
}

cudaError_t launch_plane_moments(const PlaneSelect& q, uint32_t sum_order, float* out, cudaStream_t stream) {
  if (q.n_clouds == 0) return cudaSuccess;
  if (sum_order == 0) k_plane_moments<0><<<q.n_clouds, PM_THREADS, 0, stream>>>(q, out);
  else if (sum_order == 1) k_plane_moments<1><<<q.n_clouds, PM_THREADS, 0, stream>>>(q, out);
  else k_plane_moments<2><<<q.n_clouds, PM_THREADS, 0, stream>>>(q, out);
  return cudaGetLastError();
}

}  // namespace cm
