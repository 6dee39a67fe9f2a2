// cm_cells.cuh -- the neighbour search on the sorted cell keys, shared by the radius outlier removal (cm_outlier.cu), the
// statistical outlier removal (cm_statistical.cu), the Euclidean cluster extraction (cm_cluster.cu) and the normal
// estimation (cm_normals.cu).
//
// The cloud goes through the VoxelGrid front end with a cell edge chosen by the filter (keys + onesweep sort): the points
// of one cell are one run of the sorted keys, the cells of one x-row neighbours in key order. With the edge
// radius * (1 + 2^-8), two points closer than the radius are at most one cell apart on every axis as long as
// |coordinate / cell| < 2^14 (check_cell_margin), so a query searches the 3 x 3 rows of cells around its own: nine row
// segments, each one contiguous range of sorted positions, from the cell table (k_ror_table) or from a binary search.
// The row order, the margin and the distance rounding below are what make the filters bit-equal to PCL.
#pragma once

#include <type_traits>

#include "cm_kernels.h"

namespace cm {

// sorted position j: a (key, value) uint2 record for 4-byte keys, a key array and a value array for 8-byte keys, in the
// buffers the sort's last pass wrote
template <typename KeyT>
struct Sorted {
  const void* keys;
  const uint32_t* vals;
  __device__ __forceinline__ unsigned long long key(uint32_t j) const {
    if constexpr (sizeof(KeyT) == 4) return reinterpret_cast<const uint2*>(keys)[j].x;
    else return reinterpret_cast<const unsigned long long*>(keys)[j];
  }
  __device__ __forceinline__ uint32_t val(uint32_t j) const {
    if constexpr (sizeof(KeyT) == 4) return reinterpret_cast<const uint2*>(keys)[j].y;
    else return vals[j];
  }
};

template <typename KeyT>
__device__ __forceinline__ Sorted<KeyT> sorted_of(const VoxelParams& p) {
  const bool odd = (p.info->num_passes & 1u) != 0u;
  return Sorted<KeyT>{odd ? p.keys_b : p.keys_a, odd ? p.vals_b : p.vals_a};
}

// the first of the sorted positions [0, M) whose key is >= k
template <typename KeyT>
__device__ __forceinline__ uint32_t lower_bound(const Sorted<KeyT>& s, uint32_t M, unsigned long long k) {
  uint32_t lo = 0, hi = M;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (s.key(mid) < k) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// The cell of sorted position i and its frame: several clouds in one call are frames of the key (frame f in the bits above
// idx_bits), and neighbours are only searched inside the query's own frame. False for a non-finite point (keys of frame
// >= n_frames). skip for a frame k_grid_setup could not key: its keys are all 0 but its div_b is real, so its rows would
// lie outside the cell table; the host refuses such a call before the search is enqueued, and its points are left alone.
struct QueryCell {
  unsigned long long frame, fbits, c0, c1, c2, d0, d1, d2;
};
template <typename KeyT>
__device__ __forceinline__ bool query_cell(const VoxelParams& p, const Sorted<KeyT>& s, uint32_t i, QueryCell& qc, bool& skip) {
  const uint32_t idx_bits = p.info->idx_bits;
  const unsigned long long full_key = s.key(i);
  qc.frame = idx_bits >= 64 ? 0ull : (full_key >> idx_bits);
  skip = false;
  if (qc.frame >= p.n_frames) return false;
  qc.fbits = idx_bits >= 64 ? 0ull : (qc.frame << idx_bits);
  const unsigned long long key = full_key - qc.fbits;
  const GridDev g = p.grid[qc.frame];
  if (g.zero_keys) { skip = true; return true; }
  qc.d0 = (unsigned long long)g.div_b[0]; qc.d1 = (unsigned long long)g.div_b[1]; qc.d2 = (unsigned long long)g.div_b[2];
  qc.c0 = key % qc.d0;
  const unsigned long long t = key / qc.d0;
  qc.c1 = t % qc.d1; qc.c2 = t / qc.d1;
  return true;
}

// Row segment rr of the nine, nearest first: the own row, the four rows sharing a face, the four diagonal ones (a filter
// that stops on a count is usually decided before the far rows are read). [lo, hi) of sorted positions; without the table
// hi = M and the walk stops at the first key above k_hi. False when the row lies outside the grid.
template <typename KeyT, bool TABLE>
__device__ __forceinline__ bool row_segment(const Sorted<KeyT>& s, const uint32_t* cell_start, uint32_t M, const QueryCell& qc,
                                            int rr, uint32_t& lo, uint32_t& hi, unsigned long long& k_hi) {
  // (dz + 1, dy + 1) of row rr, two bits each: (0,0) (0,-1) (0,1) (-1,0) (1,0) (-1,-1) (-1,1) (1,-1) (1,1)
  const int dz = (int)((0x28215u >> (2 * rr)) & 3u) - 1, dy = (int)((0x22161u >> (2 * rr)) & 3u) - 1;
  if ((dz < 0 && qc.c2 == 0) || (dz > 0 && qc.c2 + 1 >= qc.d2)) return false;
  if ((dy < 0 && qc.c1 == 0) || (dy > 0 && qc.c1 + 1 >= qc.d1)) return false;
  const unsigned long long x_lo = qc.c0 > 0 ? qc.c0 - 1 : 0, x_hi = qc.c0 + 1 < qc.d0 ? qc.c0 + 1 : qc.d0 - 1;
  const unsigned long long row = ((qc.c2 + dz) * qc.d1 + (qc.c1 + dy)) * qc.d0;
  const unsigned long long k_lo = qc.fbits + row + x_lo;
  k_hi = qc.fbits + row + x_hi;
  if constexpr (TABLE) {
    lo = __ldg(cell_start + k_lo);
    hi = __ldg(cell_start + k_hi + 1);
  } else {
    lo = lower_bound(s, M, k_lo);
    hi = M;
  }
  return true;
}

// FLANN's float squared distance (L2_Simple): (dx*dx + dy*dy) + dz*dz, every operation rounded on its own, never fused
__device__ __forceinline__ float flann_d2(const float4& q, const float4& d) {
  const float ex = __fsub_rn(q.x, d.x), ey = __fsub_rn(q.y, d.y), ez = __fsub_rn(q.z, d.z);
  return __fadd_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)), __fmul_rn(ez, ez));
}

// One thread of the search: the cell margin only covers |coordinate / cell| < 2^14, so a cloud that reaches further sets
// CM_DEV_E_KEY_RANGE, which the host reports as CM_E_KEY_RANGE.
__device__ __forceinline__ void check_cell_margin(const VoxelParams& p) {
  int worst = 0;
  for (uint32_t f = 0; f < p.n_frames; ++f) {
    if (p.frame_surv_start[f + 1] == p.frame_surv_start[f]) continue;
    const GridDev gf = p.grid[f];
    for (int a = 0; a < 3; ++a) worst = max(worst, max(abs(gf.min_b[a]), abs(gf.max_b[a])));
  }
  if (worst >= (1 << 14)) atomicExch(&p.ctrl->error, (uint32_t)CM_DEV_E_KEY_RANGE);
}

// f(KeyT{}) for the width of the sorted keys
template <typename F>
void with_key_type(const VoxelParams& p, F&& f) {
  if (p.key_bytes == 4) f(uint32_t{});
  else f((unsigned long long)0);
}

// f(KeyT{}, std::integral_constant<bool, TABLE>{}) for the width of the sorted keys and whether the cell table was built
template <typename F>
void with_cells(const VoxelParams& p, const uint32_t* cell_start, F&& f) {
  with_key_type(p, [&](auto key) {
    if (cell_start) f(key, std::true_type{});
    else f(key, std::false_type{});
  });
}

}  // namespace cm
