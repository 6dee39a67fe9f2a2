// cm_outlier.cu -- pcl::RadiusOutlierRemoval on the sorted cell keys for sm_100a.
//
// Replaces outlierRemoval() of the reference (pcl_preprocessing/src/pc_preprocessing_main.cpp:184-192, called from
// removeGround :119; parameters Parameter.h:23-24: radius 0.15 m, min_neighbor 1): PCL 1.8.1 builds a FLANN kd-tree over the
// cloud and, for every point, counts the points strictly inside the radius (the point itself included); a point is kept iff
// that count exceeds min_pts (`negative` inverts).
//
// Here the cloud goes through the VoxelGrid front end with a cell edge slightly above the radius (keys + onesweep sort:
// points of one cell become one run, cells of one x-row neighbours in key order), and every point then counts inside the
// 3 x 3 rows of cells around its own: nine binary searches for the row segments [x-1, x+1], a walk over each segment
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
#include "cm_kernels.h"

namespace cm {

namespace {

constexpr int ROR_THREADS = 256;

// cell_start[k] = first sorted position with key >= k, for k in [0, table_keys]. Thread i looks at sorted element i: where
// a new key run starts, the gap (previous key, this key] is filled with i by the whole warp.
template <typename KeyT>
__global__ void __launch_bounds__(ROR_THREADS) k_ror_table(const VoxelParams p, const RorParams r) {
  constexpr bool REC = sizeof(KeyT) == 4;
  const uint32_t M = p.frame_surv_start[p.n_frames];
  const uint32_t i = blockIdx.x * ROR_THREADS + threadIdx.x;
  const SortInfo si = *p.info;
  const bool odd = (si.num_passes & 1u) != 0u;
  const void* __restrict__ sorted = odd ? p.keys_b : p.keys_a;
  auto key_at = [&](uint32_t j) -> unsigned long long {
    if constexpr (REC) return reinterpret_cast<const uint2*>(sorted)[j].x;
    else return reinterpret_cast<const unsigned long long*>(sorted)[j];
  };
  const unsigned long long K = r.table_keys;
  // gap of this thread: table entries (from, to] get the value i
  unsigned long long from = 1, to = 0;  // empty
  if (i < M) {
    const unsigned long long k = min(key_at(i), K);
    if (i == 0) { from = 0; to = k; r.cell_start[0] = 0; }
    else {
      const unsigned long long kp = min(key_at(i - 1), K);
      if (k != kp) { from = kp + 1; to = k; }
    }
  } else if (i == M) {  // behind the last element: everything above the largest key
    from = M ? min(key_at(M - 1), K) + 1 : 0;
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
    for (unsigned long long k = a + lane; k <= b; k += 32) r.cell_start[k] = val;
  }
  __syncthreads();
  const int n_long = min(s_n, LIST);
  for (int g = 0; g < n_long; ++g) {
    const unsigned long long a = s_from[g], b = s_to[g];
    const uint32_t val = s_val[g];
    for (unsigned long long k = a + threadIdx.x; k <= b; k += ROR_THREADS) r.cell_start[k] = val;
  }
}

template <typename KeyT, bool TABLE>
__global__ void __launch_bounds__(ROR_THREADS) k_ror_count(const VoxelParams p, const RorParams r) {
  constexpr bool REC = sizeof(KeyT) == 4;
  const uint32_t M = p.frame_surv_start[p.n_frames];
  const uint32_t i = blockIdx.x * ROR_THREADS + threadIdx.x;
  if (i >= M) return;
  const SortInfo si = *p.info;
  const bool odd = (si.num_passes & 1u) != 0u;
  const void* __restrict__ sorted = odd ? p.keys_b : p.keys_a;
  const uint32_t* __restrict__ vals = odd ? p.vals_b : p.vals_a;
  auto key_at = [&](uint32_t j) -> unsigned long long {
    if constexpr (REC) return reinterpret_cast<const uint2*>(sorted)[j].x;
    else return reinterpret_cast<const unsigned long long*>(sorted)[j];
  };
  auto val_at = [&](uint32_t j) -> uint32_t {
    if constexpr (REC) return reinterpret_cast<const uint2*>(sorted)[j].y;
    else return vals[j];
  };
  const uint32_t idx_bits = si.idx_bits;
  const unsigned long long full_key = key_at(i);
  // several clouds in one call are frames of the key (frame f in the bits above idx_bits): neighbours are only searched
  // inside the point's own frame. Keys of frame >= n_frames: non-finite points, never kept (the mask array was cleared).
  const unsigned long long frame = idx_bits >= 64 ? 0ull : (full_key >> idx_bits);
  if (frame >= p.n_frames) return;
  const unsigned long long fbits = idx_bits >= 64 ? 0ull : (frame << idx_bits);
  const unsigned long long key = full_key - fbits;
  const GridDev g = p.grid[frame];
  // the cell margin (see the host side) only covers |coordinate / cell| < 2^14
  if (i == 0) {
    int worst = 0;
    for (uint32_t f = 0; f < p.n_frames; ++f) {
      if (p.frame_surv_start[f + 1] == p.frame_surv_start[f]) continue;
      const GridDev gf = p.grid[f];
      for (int a = 0; a < 3; ++a) worst = max(worst, max(abs(gf.min_b[a]), abs(gf.max_b[a])));
    }
    if (worst >= (1 << 14)) atomicExch(&p.ctrl->error, (uint32_t)CM_DEV_E_KEY_RANGE);
  }
  // a frame k_grid_setup could not key has every key at 0 but its real div_b: its rows would lie outside the cell table.
  // The host refuses such a call before this kernel is enqueued; its points stay unmarked here all the same.
  if (g.zero_keys) return;
  const unsigned long long d0 = (unsigned long long)g.div_b[0], d1 = (unsigned long long)g.div_b[1],
                           d2 = (unsigned long long)g.div_b[2];
  const unsigned long long c0 = key % d0, t = key / d0, c1 = t % d1, c2 = t / d1;
  const uint32_t me = val_at(i);
  const float4 q = __ldg(p.pts + me);
  const unsigned long long x_lo = c0 > 0 ? c0 - 1 : 0, x_hi = c0 + 1 < d0 ? c0 + 1 : d0 - 1;
  uint32_t cnt = 0;
  const uint32_t need = r.min_pts + 1u;  // the outcome is decided once this many neighbours were seen
  // the nine rows of cells, nearest first (own row, the four rows sharing a face, the four diagonal ones): the outcome
  // only depends on the total count, and the close rows usually decide it before the far ones are read
  for (int rr = 0; rr < 9 && cnt < need; ++rr) {
    // (dz + 1, dy + 1) of row rr, two bits each: (0,0) (0,-1) (0,1) (-1,0) (1,0) (-1,-1) (-1,1) (1,-1) (1,1)
    const int dz = (int)((0x28215u >> (2 * rr)) & 3u) - 1, dy = (int)((0x22161u >> (2 * rr)) & 3u) - 1;
    {
      if ((dz < 0 && c2 == 0) || (dz > 0 && c2 + 1 >= d2)) continue;
      if ((dy < 0 && c1 == 0) || (dy > 0 && c1 + 1 >= d1)) continue;
      const unsigned long long row = ((c2 + dz) * d1 + (c1 + dy)) * d0;
      const unsigned long long k_lo = fbits + row + x_lo, k_hi = fbits + row + x_hi;
      uint32_t lo = 0, hi = M;
      if constexpr (TABLE) {  // the row segment straight from the table
        lo = __ldg(r.cell_start + k_lo);
        hi = __ldg(r.cell_start + k_hi + 1);
      } else {                // lower bound of k_lo in the sorted keys
        while (lo < hi) {
          const uint32_t mid = (lo + hi) >> 1;
          if (key_at(mid) < k_lo) lo = mid + 1; else hi = mid;
        }
        hi = M;
      }
      for (uint32_t j = lo; j < hi && cnt < need; ++j) {
        if (!TABLE && key_at(j) > k_hi) break;
        const float4 d = __ldg(p.pts + val_at(j));
        const float ex = __fsub_rn(q.x, d.x), ey = __fsub_rn(q.y, d.y), ez = __fsub_rn(q.z, d.z);
        const float acc = __fadd_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)), __fmul_rn(ez, ez));
        if (acc < r.r2) ++cnt;
      }
    }
  }
  const bool inlier = cnt > r.min_pts;
  if (inlier != (r.negative != 0u)) r.mask[me] = (unsigned short)(1u << frame);  // zone = cloud
}

}  // namespace

cudaError_t launch_radius_table(const VoxelParams& p, const RorParams& r, cudaStream_t stream) {
  const uint32_t blocks = (p.max_points + 1 + ROR_THREADS - 1) / ROR_THREADS;  // one thread behind the last element
  if (p.key_bytes == 4) k_ror_table<uint32_t><<<blocks, ROR_THREADS, 0, stream>>>(p, r);
  else k_ror_table<unsigned long long><<<blocks, ROR_THREADS, 0, stream>>>(p, r);
  return cudaGetLastError();
}

cudaError_t launch_radius_count(const VoxelParams& p, const RorParams& r, cudaStream_t stream) {
  if (p.max_points == 0) return cudaSuccess;
  const uint32_t blocks = (p.max_points + ROR_THREADS - 1) / ROR_THREADS;
  if (r.cell_start) {
    if (p.key_bytes == 4) k_ror_count<uint32_t, true><<<blocks, ROR_THREADS, 0, stream>>>(p, r);
    else k_ror_count<unsigned long long, true><<<blocks, ROR_THREADS, 0, stream>>>(p, r);
  } else {
    if (p.key_bytes == 4) k_ror_count<uint32_t, false><<<blocks, ROR_THREADS, 0, stream>>>(p, r);
    else k_ror_count<unsigned long long, false><<<blocks, ROR_THREADS, 0, stream>>>(p, r);
  }
  return cudaGetLastError();
}

}  // namespace cm
