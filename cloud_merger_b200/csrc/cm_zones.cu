// cm_zones.cu -- zone slicing: several PassThrough chains evaluated in ONE pass over a cloud, one order-preserving
// compacted output per chain (multi-output stream compaction) for sm_100a.
//
// Replaces the per-sensor sequences of the reference that run pcl::PassThrough over the same cloud again and again
// (paths relative to timspilak/cloud_merger):
//   * getCloudPart x5 per sensor, each followed by the two z windows of removeGround
//     (pcl_preprocessing/src/pc_preprocessing_main.cpp:49-59, 80-92, 228-312): 15 PassThrough runs + copies per cloud;
//   * filter_ROI_R's three x ranges and remove_ground's two z windows (my_cloud_fusion/src/CloudFusionNode.h:145-216).
// A "zone" is a chain of up to CM_MAX_ZONE_PASSES PassThrough stages (inclusive float window, non-finite rejected,
// `negative` keeps the outside; chained stages AND together). Zones may overlap (the reference's x windows share their
// end points: a point exactly on a boundary is copied into both neighbours) and need not cover the cloud (the z windows
// leave the gap (z_max_g, z_max_g + 0.01)). Inside every zone the points keep their input order, like PassThrough.
//
// Three launches: k_zone_count (membership mask per point + per-tile counts per zone), k_zone_scan (one CTA per zone:
// per-tile offsets; the last CTA to finish lays the zones out one after the other), k_zone_scatter (ranks from warp ballots -> points and source indices to their final place).
// Roofline: HBM. Algorithmic bytes = n * (16 read + 2 mask written + 16 + 2 read again) + sum(zone sizes) * (16 + 4).
#include <cstdlib>

#include "cm_kernels.h"

namespace cm {

namespace {

constexpr int ZN_THREADS = 256;
constexpr int ZN_IPT = 4;
constexpr int ZN_TILE = ZN_THREADS * ZN_IPT;  // 1024 points per tile
constexpr int ZN_WARPS = ZN_THREADS / 32;

__device__ __forceinline__ bool zone_pass_keeps(const PassDev& ps, const float4& v) {
  const float f = ps.axis == 0 ? v.x : (ps.axis == 1 ? v.y : (ps.axis == 2 ? v.z : v.w));
  if (!finite_f32(f)) return false;
  if (!ps.negative) return !(f < ps.lo || f > ps.hi);
  return !(f >= ps.lo && f <= ps.hi);
}

// membership of one point: bit z set iff every stage of zone z keeps it (PCL 1.8.1 PassThrough::applyFilterIndices:
// a point with a non-finite x, y or z passes no stage). A zone without stages is no filter at all: it keeps every point.
__device__ __forceinline__ uint32_t zone_mask_chain(const ZoneSet& zs, const float4& v) {
  const bool fin = finite_f32(v.x) && finite_f32(v.y) && finite_f32(v.z);
  uint32_t m = 0;
  for (int z = 0; z < zs.n_zones; ++z) {
    const int np = zs.zone[z].n_pass;
    bool keep = fin || np == 0;
    for (int k = 0; k < np; ++k) keep = keep && zone_pass_keeps(zs.zone[z].pass[k], v);
    m |= (keep ? 1u : 0u) << z;
  }
  return m;
}
// Every zone is a box (ZoneSet.all_box): lo / hi of x, y, z, intensity sit in shared memory as two float4 per zone
// (+-FLT_MAX where a zone has no stage on an axis; the intensity test is skipped through no_i_mask for zones without an
// intensity stage, so that a NaN intensity only matters where PCL would look at it): two 16-byte broadcast loads and
// eight compares per zone.
__device__ __forceinline__ uint32_t zone_mask_box(const float4* s_lo, const float4* s_hi, int n_zones, uint32_t no_i_mask,
                                                  const float4& v) {
  uint32_t m = 0;
  for (int z = 0; z < n_zones; ++z) {
    const float4 lo = s_lo[z], hi = s_hi[z];
    const bool keep = (v.x >= lo.x) & (v.x <= hi.x) & (v.y >= lo.y) & (v.y <= hi.y) & (v.z >= lo.z) & (v.z <= hi.z);
    const bool keep_i = (v.w >= lo.w) & (v.w <= hi.w);
    m |= ((keep ? 1u : 0u) & ((keep_i ? 1u : 0u) | (no_i_mask >> z))) << z;
  }
  return m;
}

// GIANT: the zones are the ranks of the giant-cloud mode; the mask of a point (one bit: the rank owning its voxel index, from
// the device-resident plan) is derived here, in the sweep that counts -- no separate mask kernel and no second read.
template <bool BOX, bool GIVEN, bool GIANT = false>
__global__ void __launch_bounds__(ZN_THREADS) k_zone_count(const ZoneParams p) {
  __shared__ uint32_t s_cnt[CM_MAX_ZONES];
  __shared__ __align__(16) float4 s_lo[CM_MAX_ZONES], s_hi[CM_MAX_ZONES];
  __shared__ unsigned long long s_split[CM_MAX_ZONES];
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t n = p.n_points;
  const uint32_t tile = blockIdx.x;
  RouteGrid rg;
  if (GIANT) {
    rg = p.giant_plan->grid;
    if (tid < CM_MAX_ZONES) s_split[tid] = p.giant_plan->splitter[tid];
  }
  if (tid < CM_MAX_ZONES) {
    s_cnt[tid] = 0;
    if (BOX && (int)tid < p.zones.n_zones) {
      const ZoneDev& zd = p.zones.zone[tid];
      s_lo[tid] = make_float4(zd.lo[0], zd.lo[1], zd.lo[2], zd.lo[3]);
      s_hi[tid] = make_float4(zd.hi[0], zd.hi[1], zd.hi[2], zd.hi[3]);
    }
  }
  uint32_t no_i_mask = 0;  // bit z: zone z has no intensity stage
  if (BOX)
    for (int z = 0; z < p.zones.n_zones; ++z) no_i_mask |= (p.zones.zone[z].use_i ? 0u : 1u) << z;
  __syncthreads();
  const uint32_t base = tile * ZN_TILE + warp * (32 * ZN_IPT) + lane;
  float4 v[ZN_IPT];
#pragma unroll
  for (int i = 0; i < ZN_IPT; ++i) {
    const uint32_t g = base + 32 * i;
    v[i] = (!GIVEN && g < n) ? ldg_stream_f4(p.pts + g) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
#pragma unroll
  for (int i = 0; i < ZN_IPT; ++i) {
    const uint32_t g = base + 32 * i;
    uint32_t m = 0;
    if (g < n) {
      if (GIVEN) {
        m = p.mask[g];
      } else if (GIANT) {
        unsigned long long key;
        uint32_t dest = p.giant_invalid_part;  // non-finite points stay where they are (VoxelGrid skips them)
        if (route_key(rg, v[i], &key)) {
          dest = 0;
          for (int k = 0; k + 1 < p.zones.n_zones; ++k) dest += (key >= s_split[k]) ? 1u : 0u;
        }
        m = 1u << dest;
        p.mask[g] = (unsigned short)m;
      } else {
        m = BOX ? zone_mask_box(s_lo, s_hi, p.zones.n_zones, no_i_mask, v[i]) : zone_mask_chain(p.zones, v[i]);
        p.mask[g] = (unsigned short)m;
      }
    }
    // one shared-memory increment per zone the point belongs to (usually one); lanes of a warp that hit the same zone
    // are aggregated by the hardware (ATOMS.POPC.INC)
    while (m) {
      const uint32_t z = (uint32_t)__ffs(m) - 1u;
      m &= m - 1u;
      atomicAdd(&s_cnt[z], 1u);
    }
  }
  __syncthreads();
  if ((int)tid < p.zones.n_zones) p.tile_count[(size_t)tid * p.n_tiles + tile] = s_cnt[tid];  // zone-major
}

// One CTA per zone: exclusive scan of the zone's tile counts (offsets relative to the zone's start) and the zone total;
// the CTA that finishes last turns the totals into zone starts (zone z starts where zone z-1 ends).
__global__ void __launch_bounds__(1024) k_zone_scan(const ZoneParams p) {
  __shared__ uint32_t s_scr[33];
  __shared__ uint32_t s_run, s_last;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
  const uint32_t z = blockIdx.x;
  const uint32_t nt = p.n_tiles;
  const uint32_t* cnt = p.tile_count + (size_t)z * nt;
  uint32_t* off = p.tile_offset + (size_t)z * nt;
  if (tid == 0) s_run = 0;
  __syncthreads();
  for (uint32_t i0 = 0; i0 < nt; i0 += 1024u * 8u) {
    uint32_t c[8];
    uint32_t sum = 0;
    const uint32_t b = i0 + tid * 8u;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      c[k] = (b + k < nt) ? cnt[b + k] : 0u;
      sum += c[k];
    }
    const uint32_t incl = warp_incl_scan_u32(sum);
    if (lane == 31) s_scr[w] = incl;
    __syncthreads();
    if (w == 0) {
      const uint32_t t = s_scr[lane];
      const uint32_t ti = warp_incl_scan_u32(t);
      s_scr[lane] = ti - t;
      if (lane == 31) s_scr[32] = ti;
    }
    __syncthreads();
    uint32_t run = s_run + s_scr[w] + incl - sum;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      if (b + k < nt) off[b + k] = run;
      run += c[k];
    }
    __syncthreads();
    if (tid == 0) s_run += s_scr[32];
    __syncthreads();
  }
  if (tid == 0) {
    p.zone_total[z] = s_run;
    __threadfence();
    s_last = atomicAdd(p.scan_ticket, 1u) == gridDim.x - 1u ? 1u : 0u;
  }
  __syncthreads();
  if (s_last && tid == 0) {
    __threadfence();
    // Each zone total is at most n_points, but up to CM_MAX_ZONES of them add up past 2^32: the sum is 64-bit, and a sum
    // beyond 0xFFFFFFF0 reports the saturated 0xFFFFFFFF (more than any output may hold: the host does not regrow).
    unsigned long long run = 0;
    for (uint32_t k = 0; k < gridDim.x; ++k) {
      p.zone_begin[k] = (uint32_t)min(run, 0xFFFFFFFFull);
      run += reinterpret_cast<volatile uint32_t*>(p.zone_total)[k];
    }
    const uint32_t total = run > 0xFFFFFFF0ull ? 0xFFFFFFFFu : (uint32_t)run;
    p.zone_begin[gridDim.x] = total;
    if (run > p.out_capacity) *p.overflow = total;  // the scatter kernel then writes nothing
    *p.scan_ticket = 0;                           // ready for the next split
  }
}

template <bool REMOTE>
__global__ void __launch_bounds__(ZN_THREADS) k_zone_scatter(const ZoneParams p) {
  __shared__ uint32_t s_wcnt[ZN_WARPS][CM_MAX_ZONES];
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (*p.overflow) return;
  const uint32_t n = p.n_points;
  const uint32_t tile = blockIdx.x;
  const uint32_t base = tile * ZN_TILE + warp * (32 * ZN_IPT) + lane;
  float4 v[ZN_IPT];
  uint32_t m[ZN_IPT];
#pragma unroll
  for (int i = 0; i < ZN_IPT; ++i) {
    const uint32_t g = base + 32 * i;
    m[i] = g < n ? (uint32_t)p.mask[g] : 0u;
    v[i] = (g < n && m[i]) ? ldg_stream_f4(p.pts + g) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  // zones present in this warp's rows (lidar clouds are spatially coherent: usually one or two of them), and the warp's
  // count per zone (lane z holds zone z) for the prefix over the warps of the tile
  uint32_t present = 0;
#pragma unroll
  for (int i = 0; i < ZN_IPT; ++i) present |= __reduce_or_sync(0xFFFFFFFFu, m[i]);
  uint32_t cnt_z = 0;
  for (uint32_t zs = present; zs; zs &= zs - 1u) {
    const uint32_t z = (uint32_t)__ffs(zs) - 1u;
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < ZN_IPT; ++i) c += (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, (m[i] >> z) & 1u));
    if (lane == z) cnt_z = c;
  }
  if ((int)lane < CM_MAX_ZONES) s_wcnt[warp][lane] = cnt_z;
  __syncthreads();
  const uint32_t lt = lanemask_lt();
  for (uint32_t zs = present; zs; zs &= zs - 1u) {
    const uint32_t z = (uint32_t)__ffs(zs) - 1u;
    // REMOTE: the zone is a destination rank; its points go straight into that rank's receive buffer over NVLink
    uint32_t pos = (REMOTE ? p.zone_remote_base[z] : p.zone_begin[z]) + p.tile_offset[(size_t)z * p.n_tiles + tile];
    float4* __restrict__ dst = REMOTE ? p.zone_ptr[z] : p.out_xyzi;
    for (uint32_t w2 = 0; w2 < warp; ++w2) pos += s_wcnt[w2][z];
#pragma unroll
    for (int i = 0; i < ZN_IPT; ++i) {
      const bool in = (m[i] >> z) & 1u;
      const uint32_t b = __ballot_sync(0xFFFFFFFFu, in);
      if (in) {
        const uint32_t q = pos + (uint32_t)__popc(b & lt);
        dst[q] = v[i];
        if (!REMOTE) p.out_src[q] = base + 32 * i;
      }
      pos += (uint32_t)__popc(b);
    }
  }
}

// The exchange of the giant-cloud mode: zone z is destination rank z and its points are stored into that rank's receive
// buffer over NVLink (zone_ptr[z], from element zone_remote_base[z] + the tile's offset on). The tile is first grouped by
// destination in shared memory and then written out linearly, so that a destination receives its ~TILE / world points of the
// tile as ONE contiguous run of 16-byte stores (2 KB at world = 8) instead of the ~64-byte pieces a warp's ballot ranks
// produce: NVLink moves large writes at close to its line rate and small ones at a fraction of it.
__global__ void __launch_bounds__(ZN_THREADS) k_zone_scatter_remote(const ZoneParams p) {
  __shared__ uint32_t s_wcnt[ZN_WARPS][CM_MAX_ZONES];
  __shared__ uint32_t s_zoff[CM_MAX_ZONES + 1];  // where zone z starts in the staged tile
  __shared__ uint32_t s_zdst[CM_MAX_ZONES];      // ... and in its destination buffer
  __shared__ __align__(16) float4 s_pts[ZN_TILE];
  __shared__ unsigned char s_zone[ZN_TILE];
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (*p.overflow) return;
  const uint32_t n = p.n_points;
  const uint32_t tile = blockIdx.x;
  const int nz = p.zones.n_zones;
  const uint32_t base = tile * ZN_TILE + warp * (32 * ZN_IPT) + lane;
  float4 v[ZN_IPT];
  uint32_t m[ZN_IPT];
#pragma unroll
  for (int i = 0; i < ZN_IPT; ++i) {
    const uint32_t g = base + 32 * i;
    m[i] = g < n ? (uint32_t)p.mask[g] : 0u;
    m[i] &= 0u - m[i];  // one destination per point (the masks of the giant-cloud count sweep are one-hot already)
    v[i] = (g < n && m[i]) ? ldg_stream_f4(p.pts + g) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  uint32_t present = 0;
#pragma unroll
  for (int i = 0; i < ZN_IPT; ++i) present |= __reduce_or_sync(0xFFFFFFFFu, m[i]);
  uint32_t cnt_z = 0;
  for (uint32_t zs = present; zs; zs &= zs - 1u) {
    const uint32_t z = (uint32_t)__ffs(zs) - 1u;
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < ZN_IPT; ++i) c += (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, (m[i] >> z) & 1u));
    if (lane == z) cnt_z = c;
  }
  if ((int)lane < CM_MAX_ZONES) s_wcnt[warp][lane] = cnt_z;
  __syncthreads();
  if (warp == 0) {  // lane z: the tile's points for destination z -> start of the zone in the staged tile
    uint32_t c = 0;
    if ((int)lane < nz)
      for (int w2 = 0; w2 < ZN_WARPS; ++w2) c += s_wcnt[w2][lane];
    const uint32_t incl = warp_incl_scan_u32(c);
    if ((int)lane < nz) {
      s_zoff[lane] = incl - c;
      s_zdst[lane] = p.zone_remote_base[lane] + p.tile_offset[(size_t)lane * p.n_tiles + tile];
    }
    if ((int)lane == nz - 1) s_zoff[nz] = incl;
  }
  __syncthreads();
  const uint32_t lt = lanemask_lt();
  for (uint32_t zs = present; zs; zs &= zs - 1u) {
    const uint32_t z = (uint32_t)__ffs(zs) - 1u;
    uint32_t pos = s_zoff[z];
    for (uint32_t w2 = 0; w2 < warp; ++w2) pos += s_wcnt[w2][z];
#pragma unroll
    for (int i = 0; i < ZN_IPT; ++i) {
      const bool in = (m[i] >> z) & 1u;
      const uint32_t b = __ballot_sync(0xFFFFFFFFu, in);
      if (in) {
        const uint32_t q = pos + (uint32_t)__popc(b & lt);
        s_pts[q] = v[i];
        s_zone[q] = (unsigned char)z;
      }
      pos += (uint32_t)__popc(b);
    }
  }
  __syncthreads();
  const uint32_t total = s_zoff[nz];
  for (uint32_t q = tid; q < total; q += ZN_THREADS) {
    const uint32_t z = s_zone[q];
    p.zone_ptr[z][s_zdst[z] + (q - s_zoff[z])] = s_pts[q];
  }
}

}  // namespace

uint32_t zone_tile_points() { return ZN_TILE; }

// Only the last stage again (the counts and offsets of the previous launch_zone_split are still in place): used after
// the output arrays had to grow.
cudaError_t launch_zone_scatter(const ZoneParams& p, cudaStream_t stream) {
  if (!p.n_tiles) return cudaSuccess;
  k_zone_scatter<false><<<p.n_tiles, ZN_THREADS, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_zone_scatter_remote(const ZoneParams& p, cudaStream_t stream) {
  if (!p.n_tiles) return cudaSuccess;
  static const bool direct = getenv("CM_GIANT_DIRECT_STORES") != nullptr;  // A/B: the unstaged ballot-rank stores
  if (direct) k_zone_scatter<true><<<p.n_tiles, ZN_THREADS, 0, stream>>>(p);
  else k_zone_scatter_remote<<<p.n_tiles, ZN_THREADS, 0, stream>>>(p);
  return cudaGetLastError();
}

// rank `me`'s part of destination r starts after the parts of the ranks before it (rank order = source order)
__global__ void k_giant_offsets(const uint32_t* __restrict__ counts_all, uint32_t stride, uint32_t world, uint32_t me,
                                uint32_t* remote_base, uint32_t* overflow) {
  const uint32_t r = threadIdx.x;
  if (r >= world) return;
  uint32_t before = 0, total = 0;
  for (uint32_t s = 0; s < world; ++s) {
    const uint32_t c = counts_all[s * stride + r + 1u] - counts_all[s * stride + r];
    if (s < me) before += c;
    total += c;
  }
  remote_base[r] = before;
  const uint32_t cap = counts_all[r * stride + CM_MAX_ZONES + 1u];
  if (total > cap) atomicMax(overflow, total);
}

cudaError_t launch_giant_offsets(const uint32_t* counts_all, uint32_t stride, uint32_t world, uint32_t me, uint32_t* remote_base,
                                 uint32_t* overflow, cudaStream_t stream) {
  k_giant_offsets<<<1, 32, 0, stream>>>(counts_all, stride, world, me, remote_base, overflow);
  return cudaGetLastError();
}

cudaError_t launch_zone_count_scan(const ZoneParams& p, cudaStream_t stream) {
  if (p.n_tiles) {
    if (p.giant_plan) k_zone_count<false, false, true><<<p.n_tiles, ZN_THREADS, 0, stream>>>(p);
    else if (p.mask_given) k_zone_count<false, true><<<p.n_tiles, ZN_THREADS, 0, stream>>>(p);
    else if (p.zones.all_box) k_zone_count<true, false><<<p.n_tiles, ZN_THREADS, 0, stream>>>(p);
    else k_zone_count<false, false><<<p.n_tiles, ZN_THREADS, 0, stream>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  k_zone_scan<<<p.zones.n_zones, 1024, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_zone_split(const ZoneParams& p, cudaStream_t stream) {
  cudaError_t e = launch_zone_count_scan(p, stream);
  if (e != cudaSuccess) return e;
  if (p.n_tiles) {
    k_zone_scatter<false><<<p.n_tiles, ZN_THREADS, 0, stream>>>(p);
    e = cudaGetLastError();
  }
  return e;
}

}  // namespace cm
