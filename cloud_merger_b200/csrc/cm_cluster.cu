// cm_cluster.cu -- pcl::EuclideanClusterExtraction on the sorted cell keys for sm_100a.
//
// PCL 1.8.1 (segmentation/impl/extract_clusters.hpp, KdTreeFLANN): seeds in ascending index order, a breadth-first queue
// that adds every unprocessed neighbour (float squared distance (dx*dx + dy*dy) + dz*dz strictly below
// r2 = (float)((double)tf * tf), tf = (float)tolerance) of every queued point, clusters kept by size and then ordered by
// std::sort over reverse iterators. Its clusters are exactly the connected components of the neighbour graph, each with
// its smallest index as the seed (DESIGN section 8), so here:
//  * the cloud goes through the radius outlier removal's front end with cell edge tf * (1 + 2^-8) (keys + onesweep sort +
//    cell table): two neighbours are at most one cell apart on every axis;
//  * k_ec_gather puts the points into sorted order and sets every point's parent to itself;
//  * k_ec_hook walks the 3 x 3 rows of cells of cm_cells.cuh from every sorted position i, tests the candidates behind i
//    (one direction per pair) with FLANN's float distance, and unions the two points' trees: a parallel union-find in
//    input-index space in the style of ECL-CC, the larger root hooked under the smaller one with atomicCAS, path halving in
//    find. A root only ever gets a smaller parent, so the final root of a component is its smallest index -- PCL's seed --
//    whatever the thread timing;
//  * k_ec_label writes every finite point's root into a label array and counts the points of every root; k_ec_roots marks the
//    roots whose size is inside [min_size, max_size] in the zone-slicing mask (zone = cloud), and the zone compaction
//    lists them in ascending order: seed order. The host reads their sizes and runs PCL's std::sort on them;
//  * k_ec_keys keys every point by its cluster's output rank (the points of no kept cluster by the largest key), and a
//    stable LSD radix sort of (rank, input index) (k_ec_digits / k_ec_offsets / k_ec_scatter, 8 bits a pass) leaves every
//    cluster's indices ascending; k_ec_gather_out copies the coordinates.
#include "cm_cells.cuh"

namespace cm {

namespace {

constexpr int EC_THREADS = 256;
constexpr int RS_WARPS = 8;
constexpr int RS_ROUNDS = 16;                        // 32 keys a round per warp
constexpr uint32_t RS_TILE = RS_WARPS * 32 * RS_ROUNDS;  // keys per CTA of a radix pass
constexpr uint32_t NONE = 0xFFFFFFFFu;
constexpr uint32_t FULL = 0xFFFFFFFFu;

template <typename KeyT>
__global__ void __launch_bounds__(EC_THREADS) k_ec_gather(const VoxelParams p, float4* __restrict__ sorted_pts,
                                                          uint32_t* __restrict__ parent) {
  const uint32_t M = p.frame_surv_start[p.n_frames];
  const uint32_t i = blockIdx.x * EC_THREADS + threadIdx.x;
  if (i >= M) return;
  sorted_pts[i] = __ldg(p.pts + sorted_of<KeyT>(p).val(i));
  parent[i] = i;
}

__device__ __forceinline__ uint32_t vload(const uint32_t* a) { return *reinterpret_cast<const volatile uint32_t*>(a); }

// Root of x. Every parent is an ancestor with a smaller index, so the shortcut stores (path halving) only ever replace a
// parent by a smaller ancestor, and a racing store of another thread leaves an ancestor there as well.
__device__ __forceinline__ uint32_t ec_find(uint32_t* parent, uint32_t x) {
  uint32_t cur = vload(parent + x);
  if (cur != x) {
    uint32_t prev = x, next;
    while (cur > (next = vload(parent + cur))) {
      *reinterpret_cast<volatile uint32_t*>(parent + prev) = next;
      prev = cur;
      cur = next;
    }
  }
  return cur;
}

// the larger root goes under the smaller one; a root that was hooked meanwhile is followed to its new root
__device__ __forceinline__ void ec_union(uint32_t* parent, uint32_t a, uint32_t b) {
  uint32_t ra = ec_find(parent, a), rb = ec_find(parent, b);
  while (ra != rb) {
    if (ra > rb) { const uint32_t t = ra; ra = rb; rb = t; }
    const uint32_t old = atomicCAS(parent + rb, rb, ra);
    if (old == rb) return;
    rb = ec_find(parent, old);
    ra = ec_find(parent, ra);
  }
}

template <typename KeyT, bool TABLE>
__global__ void __launch_bounds__(EC_THREADS) k_ec_hook(const VoxelParams p, const EcParams e) {
  const uint32_t M = p.frame_surv_start[p.n_frames];
  const uint32_t i = blockIdx.x * EC_THREADS + threadIdx.x;
  if (i >= M) return;
  const Sorted<KeyT> s = sorted_of<KeyT>(p);
  // query_cell written out, so that the margin check sits between the frame and the cell decode: next to a query_cell
  // call ptxas gives 40 registers to the three instantiations that get 32 here (DESIGN section 4)
  const uint32_t idx_bits = p.info->idx_bits;
  const unsigned long long full_key = s.key(i);
  QueryCell qc;
  qc.frame = idx_bits >= 64 ? 0ull : (full_key >> idx_bits);
  if (qc.frame >= p.n_frames) return;  // a non-finite point belongs to no cluster
  qc.fbits = idx_bits >= 64 ? 0ull : (qc.frame << idx_bits);
  const unsigned long long key = full_key - qc.fbits;
  const GridDev g = p.grid[qc.frame];
  if (i == 0) check_cell_margin(p);
  if (g.zero_keys) return;  // the host refuses such a call before this kernel is enqueued
  qc.d0 = (unsigned long long)g.div_b[0]; qc.d1 = (unsigned long long)g.div_b[1]; qc.d2 = (unsigned long long)g.div_b[2];
  qc.c0 = key % qc.d0;
  const unsigned long long t = key / qc.d0;
  qc.c1 = t % qc.d1; qc.c2 = t / qc.d1;
  const float4 q = e.sorted_pts[i];
  uint32_t me = NONE;
  for (int rr = 0; rr < 9; ++rr) {
    uint32_t lo, hi;
    unsigned long long k_hi;
    if (!row_segment<KeyT, TABLE>(s, e.cell_start, M, qc, rr, lo, hi, k_hi)) continue;
    // only the candidates behind i: every pair is tested once, from its earlier sorted position
    for (uint32_t j = max(lo, i + 1); j < hi; ++j) {
      if (!TABLE && s.key(j) > k_hi) break;
      if (flann_d2(q, e.sorted_pts[j]) < e.r2) {
        if (me == NONE) me = s.val(i);
        ec_union(e.parent, me, s.val(j));
      }
    }
  }
}

__device__ __forceinline__ bool finite_xyz(const float4& v) {
  return finite_f32(v.x) && finite_f32(v.y) && finite_f32(v.z);
}

// label[i] = the root of every finite point (NONE for the others), and the points of every root. The labels go to an
// array of their own: the path-halving stores of the other threads' finds may still replace parent[i] by an ancestor
// that is not the root.
__global__ void __launch_bounds__(EC_THREADS) k_ec_label(const EcParams e, uint32_t n) {
  const uint32_t i = blockIdx.x * EC_THREADS + threadIdx.x;
  if (i >= n) return;
  if (!finite_xyz(__ldg(e.pts + i))) { e.label[i] = NONE; return; }
  const uint32_t r = ec_find(e.parent, i);
  e.label[i] = r;
  atomicAdd(e.size + r, 1u);
}

// the kept roots: bit c of the zone mask for a root of cloud c whose size is inside [min_size, max_size]
__global__ void __launch_bounds__(EC_THREADS) k_ec_roots(const EcParams e, uint32_t n) {
  const uint32_t i = blockIdx.x * EC_THREADS + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = e.size[i];
  const bool kept = e.parent[i] == i && s > 0 && s >= e.min_size && s <= e.max_size;
  uint32_t c = 0;
  while (i >= e.begin[c + 1]) ++c;
  e.mask[i] = kept ? (unsigned short)(1u << c) : (unsigned short)0;
}

// sizes of the listed roots (seed order)
__global__ void __launch_bounds__(EC_THREADS) k_ec_sizes(const EcParams e, const uint32_t* __restrict__ roots,
                                                         uint32_t n_roots, uint32_t* __restrict__ out) {
  const uint32_t k = blockIdx.x * EC_THREADS + threadIdx.x;
  if (k < n_roots) out[k] = e.size[roots[k]];
}

// rank[root] = output rank of the kept cluster at seed position k (rank may alias size: the sizes were read before)
__global__ void __launch_bounds__(EC_THREADS) k_ec_rank(const uint32_t* __restrict__ roots, const uint32_t* __restrict__ perm,
                                                        uint32_t n_roots, uint32_t* __restrict__ rank) {
  const uint32_t k = blockIdx.x * EC_THREADS + threadIdx.x;
  if (k < n_roots) rank[roots[k]] = perm[k];
}

// sort key of every point: its cluster's output rank, or n_clusters for a point of no kept cluster
__global__ void __launch_bounds__(EC_THREADS) k_ec_keys(const EcParams e, uint32_t n, uint32_t n_clusters,
                                                        const uint32_t* __restrict__ rank, uint32_t* __restrict__ keys,
                                                        uint32_t* __restrict__ vals) {
  const uint32_t i = blockIdx.x * EC_THREADS + threadIdx.x;
  if (i >= n) return;
  const uint32_t r = e.label[i];
  keys[i] = r != NONE && e.mask[r] ? rank[r] : n_clusters;
  vals[i] = i;
}

// ---- stable LSD radix sort of (key, value), 8 bits a pass ----------------------------------------------------------------
// counts[d * n_tiles + t] = keys of digit d in tile t
__global__ void __launch_bounds__(RS_WARPS * 32) k_ec_digits(const uint32_t* __restrict__ keys, uint32_t n, uint32_t shift,
                                                             uint32_t* __restrict__ counts) {
  __shared__ uint32_t s_cnt[256];
  const uint32_t tid = threadIdx.x, t = blockIdx.x, n_tiles = gridDim.x;
  s_cnt[tid] = 0;
  __syncthreads();
  const uint32_t b = t * RS_TILE, e = min(n, b + RS_TILE);
  for (uint32_t i = b + tid; i < e; i += RS_WARPS * 32) atomicAdd(&s_cnt[(keys[i] >> shift) & 255u], 1u);
  __syncthreads();
  counts[tid * n_tiles + t] = s_cnt[tid];
}

// exclusive scan of counts in place (digit-major: the first position of digit d in tile t), one CTA
__global__ void __launch_bounds__(1024) k_ec_offsets(uint32_t* __restrict__ counts, uint32_t total) {
  __shared__ uint32_t s_sum[1024];
  const uint32_t tid = threadIdx.x;
  const uint32_t per = (total + 1023) / 1024, b = min(total, tid * per), e = min(total, b + per);
  uint32_t s = 0;
  for (uint32_t i = b; i < e; ++i) s += counts[i];
  s_sum[tid] = s;
  __syncthreads();
  for (uint32_t o = 1; o < 1024; o <<= 1) {
    const uint32_t v = tid >= o ? s_sum[tid - o] : 0u;
    __syncthreads();
    s_sum[tid] += v;
    __syncthreads();
  }
  uint32_t run = s_sum[tid] - s;
  for (uint32_t i = b; i < e; ++i) {
    const uint32_t c = counts[i];
    counts[i] = run;
    run += c;
  }
}

// Every warp ranks its 512 keys in order, 32 at a time (peers of the same digit by __match_any_sync, earlier lanes first);
// the warps' digit counts are then stacked in warp order, so the pass keeps the input order of equal digits.
__global__ void __launch_bounds__(RS_WARPS * 32) k_ec_scatter(const uint32_t* __restrict__ keys_in,
                                                              const uint32_t* __restrict__ vals_in, uint32_t n, uint32_t shift,
                                                              const uint32_t* __restrict__ offsets,
                                                              uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out) {
  __shared__ uint32_t s_cnt[RS_WARPS][256];
  const uint32_t tid = threadIdx.x, w = tid >> 5, lane = tid & 31u, t = blockIdx.x, n_tiles = gridDim.x;
  for (uint32_t k = tid; k < RS_WARPS * 256; k += RS_WARPS * 32) (&s_cnt[0][0])[k] = 0;
  __syncthreads();
  const uint32_t base = t * RS_TILE + w * 32 * RS_ROUNDS;
  uint32_t dig[RS_ROUNDS], loc[RS_ROUNDS];
#pragma unroll
  for (int r = 0; r < RS_ROUNDS; ++r) {
    const uint32_t i = base + (uint32_t)r * 32u + lane;
    const uint32_t d = i < n ? (keys_in[i] >> shift) & 255u : 256u;
    const uint32_t peers = __match_any_sync(FULL, d);
    const uint32_t before = __popc(peers & ((1u << lane) - 1u));
    dig[r] = d;
    loc[r] = d < 256u ? s_cnt[w][d] + before : 0u;
    __syncwarp();
    if (d < 256u && before == 0) s_cnt[w][d] += __popc(peers);
    __syncwarp();
  }
  __syncthreads();
  {  // per digit (thread tid): the warps' counts -> the first position of each warp's keys inside the tile's digit run
    uint32_t run = 0;
    for (int ww = 0; ww < RS_WARPS; ++ww) {
      const uint32_t c = s_cnt[ww][tid];
      s_cnt[ww][tid] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < RS_ROUNDS; ++r) {
    const uint32_t i = base + (uint32_t)r * 32u + lane, d = dig[r];
    if (d >= 256u) continue;
    const uint32_t pos = offsets[d * n_tiles + t] + s_cnt[w][d] + loc[r];
    keys_out[pos] = keys_in[i];
    vals_out[pos] = vals_in[i];
  }
}

__global__ void __launch_bounds__(EC_THREADS) k_ec_gather_out(const float4* __restrict__ pts, const uint32_t* __restrict__ idx,
                                                              uint32_t n, float4* __restrict__ out) {
  const uint32_t k = blockIdx.x * EC_THREADS + threadIdx.x;
  if (k < n) out[k] = __ldg(pts + idx[k]);
}

uint32_t blocks_of(uint32_t n) { return (n + EC_THREADS - 1) / EC_THREADS; }

}  // namespace

uint32_t ec_sort_tiles(uint32_t n) { return (n + RS_TILE - 1) / RS_TILE; }

cudaError_t launch_ec_hook(const VoxelParams& p, const EcParams& e, float4* sorted_pts, cudaStream_t stream) {
  if (p.max_points == 0) return cudaSuccess;
  const uint32_t blocks = blocks_of(p.max_points);
  with_key_type(p, [&](auto key) {
    k_ec_gather<decltype(key)><<<blocks, EC_THREADS, 0, stream>>>(p, sorted_pts, e.parent);
  });
  with_cells(p, e.cell_start, [&](auto key, auto table) {
    k_ec_hook<decltype(key), decltype(table)::value><<<blocks, EC_THREADS, 0, stream>>>(p, e);
  });
  return cudaGetLastError();
}

cudaError_t launch_ec_roots(const EcParams& e, uint32_t n, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  k_ec_label<<<blocks_of(n), EC_THREADS, 0, stream>>>(e, n);
  k_ec_roots<<<blocks_of(n), EC_THREADS, 0, stream>>>(e, n);
  return cudaGetLastError();
}

cudaError_t launch_ec_sizes(const EcParams& e, const uint32_t* roots, uint32_t n_roots, uint32_t* out, cudaStream_t stream) {
  if (n_roots == 0) return cudaSuccess;
  k_ec_sizes<<<blocks_of(n_roots), EC_THREADS, 0, stream>>>(e, roots, n_roots, out);
  return cudaGetLastError();
}

int launch_ec_order(const EcParams& e, const EcOrder& o, uint32_t n, cudaStream_t stream, cudaError_t* err) {
  *err = cudaSuccess;
  if (n == 0 || o.n_clusters == 0) return 0;
  int launches = 0;
  k_ec_rank<<<blocks_of(o.n_clusters), EC_THREADS, 0, stream>>>(o.roots, o.perm, o.n_clusters, o.rank);
  k_ec_keys<<<blocks_of(n), EC_THREADS, 0, stream>>>(e, n, o.n_clusters, o.rank, o.keys[0], o.vals[0]);
  launches += 2;
  const uint32_t tiles = ec_sort_tiles(n);
  for (uint32_t ps = 0; ps < o.passes; ++ps) {
    const uint32_t in = ps & 1u, out = in ^ 1u;
    k_ec_digits<<<tiles, RS_WARPS * 32, 0, stream>>>(o.keys[in], n, 8u * ps, o.counts);
    k_ec_offsets<<<1, 1024, 0, stream>>>(o.counts, tiles * 256u);
    k_ec_scatter<<<tiles, RS_WARPS * 32, 0, stream>>>(o.keys[in], o.vals[in], n, 8u * ps, o.counts, o.keys[out], o.vals[out]);
    launches += 3;
  }
  k_ec_gather_out<<<blocks_of(o.n_points_out), EC_THREADS, 0, stream>>>(e.pts, o.vals[o.passes & 1u], o.n_points_out, o.out_xyzi);
  ++launches;
  *err = cudaGetLastError();
  return launches;
}

}  // namespace cm
