// cm_outlier.cu -- pcl::RadiusOutlierRemoval on the sorted cell keys for sm_100a.
//
// Replaces outlierRemoval() of the reference (pcl_preprocessing/src/pc_preprocessing_main.cpp:184-192, called from
// removeGround :119; parameters Parameter.h:23-24: radius 0.15 m, min_neighbor 1): PCL 1.8.1 builds a FLANN kd-tree over the
// cloud and, for every point, counts the points strictly inside the radius (the point itself included); a point is kept iff
// that count exceeds min_pts (`negative` inverts).
//
// Here the cloud goes through the VoxelGrid front end with a cell edge slightly above the radius (keys + onesweep sort:
// points of one cell become one run, cells of one x-row neighbours in key order), and every point then counts inside the
// 3 x 3 rows of cells around its own (the search of cm_cells.cuh): nine binary searches for the row segments [x-1, x+1], a walk over each segment
// with the squared distance in FLANN's float order ((dx*dx + dy*dy) + dz*dz, never fused), and an early exit as soon as
// the count decides the outcome. The keep flags go to the zone-slicing mask array, whose scan + scatter kernels then
// compact the survivors in input order (cm_zones.cu).
//
// When the key space is small enough (frames << idx_bits <= 2^25, the usual case for a cropped cloud) a direct-address
// table replaces the binary searches: k_ror_table writes, for every key k, the first sorted position whose key is >= k
// (the heads of the key runs fill the gap up to their key, a warp per gap), and a row segment [k_lo, k_hi] is then just
// [cell_start[k_lo], cell_start[k_hi + 1]) -- two loads instead of ~22 dependent ones per row.
//
// Roofline: HBM/L2 for the gathers; algorithmic bytes ~ n * (8 record + 16 point) * (neighbours visited).
#include "cm_cells.cuh"

namespace cm {

namespace {

constexpr int ROR_THREADS = 256;

// cell_start[k] = first sorted position with key >= k, for k in [0, table_keys]. Thread i looks at sorted element i: where
// a new key run starts, the gap (previous key, this key] is filled with i by the whole warp.
template <typename KeyT>
__global__ void __launch_bounds__(ROR_THREADS) k_ror_table(const VoxelParams p, const CellTable t) {
  const uint32_t M = p.frame_surv_start[p.n_frames];
  const uint32_t i = blockIdx.x * ROR_THREADS + threadIdx.x;
  const Sorted<KeyT> s = sorted_of<KeyT>(p);
  const unsigned long long K = t.table_keys;
  // gap of this thread: table entries (from, to] get the value i
  unsigned long long from = 1, to = 0;  // empty
  if (i < M) {
    const unsigned long long k = min(s.key(i), K);
    if (i == 0) { from = 0; to = k; t.cell_start[0] = 0; }
    else {
      const unsigned long long kp = min(s.key(i - 1), K);
      if (k != kp) { from = kp + 1; to = k; }
    }
  } else if (i == M) {  // behind the last element: everything above the largest key
    from = M ? min(s.key(M - 1), K) + 1 : 0;
    to = K;
  }
  // short gaps: the warp of the head fills them; long ones (empty regions of the key space, the space between two
  // clouds' cell ranges) go to a list in shared memory and are filled by the whole CTA
  constexpr unsigned long long LONG_GAP = 2048;
  constexpr int LIST = 32;
  __shared__ unsigned long long s_from[LIST], s_to[LIST];
  __shared__ uint32_t s_val[LIST];
  __shared__ int s_n;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u;
  if (from <= to && to - from >= LONG_GAP) {
    const int slot = atomicAdd(&s_n, 1);
    if (slot < LIST) { s_from[slot] = from; s_to[slot] = to; s_val[slot] = i; from = 1; to = 0; }
  }
  uint32_t todo = __ballot_sync(0xffffffffu, from <= to);
  while (todo) {
    const int src = __ffs(todo) - 1;
    todo &= todo - 1;
    const unsigned long long a = __shfl_sync(0xffffffffu, from, src), b = __shfl_sync(0xffffffffu, to, src);
    const uint32_t val = __shfl_sync(0xffffffffu, i, src);
    for (unsigned long long k = a + lane; k <= b; k += 32) t.cell_start[k] = val;
  }
  __syncthreads();
  const int n_long = min(s_n, LIST);
  for (int g = 0; g < n_long; ++g) {
    const unsigned long long a = s_from[g], b = s_to[g];
    const uint32_t val = s_val[g];
    for (unsigned long long k = a + threadIdx.x; k <= b; k += ROR_THREADS) t.cell_start[k] = val;
  }
}

template <typename KeyT, bool TABLE>
__global__ void __launch_bounds__(ROR_THREADS) k_ror_count(const VoxelParams p, const RorParams r) {
  const uint32_t M = p.frame_surv_start[p.n_frames];
  const uint32_t i = blockIdx.x * ROR_THREADS + threadIdx.x;
  if (i >= M) return;
  const Sorted<KeyT> s = sorted_of<KeyT>(p);
  if (i == 0) check_cell_margin(p);
  QueryCell qc;
  bool skip;
  // a non-finite point is never kept (the mask array was cleared)
  if (!query_cell<KeyT>(p, s, i, qc, skip) || skip) return;
  const uint32_t me = s.val(i);
  const float4 q = __ldg(p.pts + me);
  uint32_t cnt = 0;
  const uint32_t need = r.min_pts + 1u;  // the outcome is decided once this many neighbours were seen
  for (int rr = 0; rr < 9 && cnt < need; ++rr) {
    uint32_t lo, hi;
    unsigned long long k_hi;
    if (!row_segment<KeyT, TABLE>(s, r.cell_start, M, qc, rr, lo, hi, k_hi)) continue;
    for (uint32_t j = lo; j < hi && cnt < need; ++j) {
      if (!TABLE && s.key(j) > k_hi) break;
      if (flann_d2(q, __ldg(p.pts + s.val(j))) < r.r2) ++cnt;
    }
  }
  const bool inlier = cnt > r.min_pts;
  if (inlier != (r.negative != 0u)) r.mask[me] = (unsigned short)(1u << qc.frame);  // zone = cloud
}

}  // namespace

cudaError_t launch_radius_table(const VoxelParams& p, const CellTable& t, cudaStream_t stream) {
  const uint32_t blocks = (p.max_points + 1 + ROR_THREADS - 1) / ROR_THREADS;  // one thread behind the last element
  with_key_type(p, [&](auto key) { k_ror_table<decltype(key)><<<blocks, ROR_THREADS, 0, stream>>>(p, t); });
  return cudaGetLastError();
}

cudaError_t launch_radius_count(const VoxelParams& p, const RorParams& r, cudaStream_t stream) {
  if (p.max_points == 0) return cudaSuccess;
  const uint32_t blocks = (p.max_points + ROR_THREADS - 1) / ROR_THREADS;
  with_cells(p, r.cell_start, [&](auto key, auto table) {
    k_ror_count<decltype(key), decltype(table)::value><<<blocks, ROR_THREADS, 0, stream>>>(p, r);
  });
  return cudaGetLastError();
}

}  // namespace cm
