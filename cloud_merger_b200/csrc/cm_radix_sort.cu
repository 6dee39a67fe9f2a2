// cm_radix_sort.cu -- in-house onesweep LSD radix sort of (voxel key, point index) pairs for sm_100a.
//
// Replaces the std::sort(index_vector) at the heart of pcl::VoxelGrid::applyFilter (PCL 1.8.1 voxel_grid.hpp, reached
// from the reference's voxelgrid(), pc_preprocessing_main.cpp:168-177). No CUB / Thrust.
//
// One launch per digit (8 bits; the top digit of a fused-key run sorted frame by frame may take up to 384 values, see
// sort_digit). The digit histograms of all passes were produced up front by k_voxel_key_hist, so a pass
// is a single sweep: each CTA takes a tile, ranks its keys by digit (ballot-based match, stable), obtains for
// each of the 256 digits the global position of its first key of that digit (chained scan; see "scanner CTAs"), and
// scatters keys and values to their final place of this pass through shared memory so that global stores are
// digit-contiguous. The number of passes is decided on the device (SortInfo.num_passes, from the significant key bits); a
// pass beyond it returns immediately, and every kernel derives the ping-pong buffer it reads from the pass number.
//
// Batches of several frames can be sorted frame by frame inside the same launches (SEG instantiations: frame-aligned tiles,
// per-frame first positions, scanners that restart at frame starts) -- the frame bits of the key then need no pass at all;
// see scanner_cta and DESIGN.md "Frame-segmented sort".
//
// Record layout in HBM: 32-bit keys travel as 8-byte (key, value) records in keys_a / keys_b (one 8-byte load and one
// 8-byte store per item and pass, digit runs of 128 bytes on average); 64-bit keys travel as separate key and value
// arrays (keys_*, vals_*).
//
// The kernel is instruction-issue bound before it is HBM bound, so the per-item instruction count is what was designed:
//   load 1, digit 1, match 24 (R2P + 8 VOTE + 8 predicated NOT + 4 three-input OR), rank 8 (one LDS, one predicated STS
//   on a warp-private counter row, one POPC), shared-memory placement 5, scatter 8  ~= 50 per item (was ~150).
//
// Roofline: HBM. Algorithmic bytes per pass = n * 2 * (key_bytes + 4).
#include <cstdio>
#include <cstdlib>

#include "cm_kernels.h"

namespace cm {

namespace {

// Shape of a worker CTA (overridable for experiments): threads, keys per thread (32-bit / 64-bit keys), CTAs per SM.
// Measured on B200, cfg2 batch, ms for the four passes: 256x16x3 0.311-0.323, 512x8x2 0.352, 320x14x2 0.324, 384x12x2 0.302;
// publishing the digit counts before the ranking (RS_EARLY_COUNT) cost more than the shorter row wait returned (0.32).
#ifndef RS_THREADS_CFG
#define RS_THREADS_CFG 384
#endif
#ifndef RS_IPT32
#define RS_IPT32 12
#endif
#ifndef RS_IPT64
#define RS_IPT64 8
#endif
#ifndef RS_MIN_CTAS
#define RS_MIN_CTAS 2
#endif
#ifndef RS_EARLY_COUNT
#define RS_EARLY_COUNT 0
#endif
constexpr int RS_THREADS = RS_THREADS_CFG;
static_assert(RS_THREADS >= CM_RADIX && RS_THREADS % 32 == 0, "one thread per digit is needed");
constexpr int RS_WARPS = RS_THREADS / 32;

template <typename KeyT>
struct SortCfg;
template <>
struct SortCfg<uint32_t> {
  static constexpr int IPT = RS_IPT32;
};
template <>
struct SortCfg<unsigned long long> {
  static constexpr int IPT = RS_IPT64;
};

// ---- scanner CTAs -------------------------------------------------------------------------------------------------------
// The first RS_SCANNERS CTAs of a pass do not sort. Rows of 256 look-back words are indexed -1 .. n_tiles-1; worker
// tile t publishes its 256 digit counts in row t, and needs, per digit, the global position of its first key of that
// digit = (number of keys with a smaller digit in the whole input) + (keys of that digit in tiles < t). The scanners
// produce exactly that number and overwrite every row with it, so a worker reads one row -- row t-1 -- instead of
// walking back over every tile in flight (that walk, 256 digits x dozens of rows per tile, cost as much L2 bandwidth as
// the keys themselves).
//
// Scanner h owns 32 consecutive digits, one per lane. Its warps take 32-row batches round-robin (warp q: batches q,
// q+8, ...) and work on them independently: poll the batch's rows (all loads of a round in flight together) until
// every count is published, prefix them in registers -- and only then enter the serial part, a shared-memory hand-over
// of the running sum from the warp of the previous batch (one 8-byte word per digit carrying the batch sequence
// number; ~100 cycles per batch). So 256 rows are being collected at any time and the serial chain of a pass is
// n_tiles/32 short hops, not n_tiles/64 global-memory round trips as in the first version (where a worker spent 43% of
// its life waiting for its row). The running sum starts from the exclusive scan of the pass's global digit histogram
// (row -1). Scanners are CTAs 0..7 of the grid, i.e. resident before any worker; workers publish their counts before
// they wait, so the pair cannot deadlock.
constexpr int RS_SCAN_DIGITS = 32;                      // one digit per lane
constexpr int RS_SCANNERS = CM_RADIX / RS_SCAN_DIGITS;  // 8 (a pass of NB bins has NB / 32)
constexpr int RS_SCAN_ROWS = 32;                        // rows per batch (one warp)
constexpr int RS_SCAN_GROUP = RS_THREADS >= 512 ? 8 : 16;  // rows polled together (register budget of the CTA shape)
static_assert(RS_THREADS >= (int)CM_WIDE_BINS, "one thread per digit of a wide pass is needed");

//
// SEG (frame-segmented sort): the tiles are frame-aligned and every frame is a sort of its own, so the running sum restarts
// at the first tile of a frame from that frame's own first positions (seg_base: frame start + exclusive scan of the frame's
// digit counts, prepared by k_seg_base); a worker on the first tile of a frame reads them itself and waits for nobody.
// NB: bins of the pass (256; CM_WIDE_BINS for the wide top digit of a SEG run): rows are NB words wide, NB / 32 scanners.
template <bool SEG, int NB = CM_RADIX>
__device__ __forceinline__ void scanner_cta(uint32_t scanner /* 0 .. NB/32-1 */, unsigned long long* rows /* row 0 */,
                                            uint32_t n_tiles, uint32_t epoch, const uint32_t* hist /* this pass */,
                                            uint32_t* err, uint32_t* s_scan, uint32_t* s_tmp /* >= 256 words */,
                                            unsigned long long* s_chain /* 32 */, const SegTile* __restrict__ seg_tile,
                                            const uint32_t* __restrict__ seg_base /* [frame][CM_SEG_PASSES][256], at this pass */) {
  const uint32_t tid = threadIdx.x, lane = tid & 31u, q = tid >> 5;
  static_assert(SEG || NB == CM_RADIX, "a wide top digit is only ranked frame by frame");
  const uint32_t d = scanner * RS_SCAN_DIGITS + lane;  // digit
  if (SEG) {
    if (q == 0) s_chain[lane] = 0ull;  // sequence number 0; the value is never used (tile 0 starts a frame)
  } else {
    // exclusive scan of the global digit histogram: where digit d starts in the output of this pass
    uint32_t tot;
    const uint32_t gb = block_excl_scan_256(tid < CM_RADIX ? hist[tid] : 0u, s_scan, &tot);
    if (tid < CM_RADIX) s_tmp[tid] = gb;
    __syncthreads();
    if (q == 0) {
      const uint32_t run0 = s_tmp[d];
      st_cg_u64(rows - CM_RADIX + d, lb_pack(epoch, CM_LB_INCL, run0));  // row -1
      s_chain[lane] = (unsigned long long)run0;                           // sequence number 0: the sum before batch 0
    }
  }
  __syncthreads();
  const uint32_t n_batches = (n_tiles + RS_SCAN_ROWS - 1) / RS_SCAN_ROWS;
  volatile unsigned long long* chain = s_chain + lane;
  for (uint32_t b = q; b < n_batches; b += RS_WARPS) {
    const uint32_t r0 = b * RS_SCAN_ROWS;
    unsigned long long* const base = rows + (size_t)r0 * NB + d;
    uint32_t c[RS_SCAN_ROWS];
#pragma unroll
    for (int g0 = 0; g0 < RS_SCAN_ROWS; g0 += RS_SCAN_GROUP) {
      uint32_t spins = 0;
      unsigned long long wd0 = 0ull;
      while (true) {
        unsigned long long w[RS_SCAN_GROUP];
#pragma unroll
        for (int k = 0; k < RS_SCAN_GROUP; ++k)
          w[k] = (r0 + g0 + k < n_tiles) ? ld_cg_u64(base + (size_t)(g0 + k) * NB) : lb_pack(epoch, CM_LB_AGG, 0u);
        bool all = true;
#pragma unroll
        for (int k = 0; k < RS_SCAN_GROUP; ++k) {
          all = all && lb_ready(w[k], epoch);
          c[g0 + k] = (uint32_t)w[k];
        }
        if (__all_sync(0xFFFFFFFFu, all)) break;
        // watchdog (wall clock): raise the device error and let everything drain
        if (__any_sync(0xFFFFFFFFu, watchdog_expired(spins, wd0))) {
          atomicExch(err, (uint32_t)CM_DEV_E_INTERNAL);
          break;
        }
        if (spins > 8) __nanosleep(50);
      }
    }
    uint32_t sum = 0;
    uint32_t abs_from = RS_SCAN_ROWS;  // SEG: rows from here on carry absolute positions (a frame started inside the batch)
    if (SEG) {
      const uint32_t mine = (r0 + lane < n_tiles) ? __ldg(&seg_tile[r0 + lane].frame) : 0u;  // lane k: row r0 + k
      const uint32_t firsts = __ballot_sync(0xFFFFFFFFu, (mine & CM_SEG_FIRST) != 0u);
      if (firsts) abs_from = (uint32_t)__ffs(firsts) - 1u;
#pragma unroll
      for (int k = 0; k < RS_SCAN_ROWS; ++k) {
        if (firsts & (1u << k)) {  // warp-uniform
          const uint32_t f = __shfl_sync(0xFFFFFFFFu, mine, k) & ~CM_SEG_FIRST;
          sum = __ldg(seg_base + (size_t)f * (CM_SEG_PASSES * CM_RADIX) + d);
        }
        sum += c[k];
        c[k] = sum;
      }
    } else {
#pragma unroll
      for (int k = 0; k < RS_SCAN_ROWS; ++k) {
        sum += c[k];
        c[k] = sum;  // inclusive within the batch
      }
    }
    // serial part: take the running sum from the previous batch's warp, pass it on
    unsigned long long x = *chain;
    uint32_t spins = 0;
    unsigned long long wd0 = 0ull;
    while ((uint32_t)(x >> 32) != b) {
      if (watchdog_expired(spins, wd0)) {
        atomicExch(err, (uint32_t)CM_DEV_E_INTERNAL);
        break;
      }
      x = *chain;
    }
    const uint32_t run = (uint32_t)x;
    if (SEG) {
      *chain = ((unsigned long long)(b + 1u) << 32) | (unsigned long long)(abs_from < RS_SCAN_ROWS ? sum : run + sum);
#pragma unroll
      for (int k = 0; k < RS_SCAN_ROWS; ++k)
        if (r0 + k < n_tiles)
          st_cg_u64(base + (size_t)k * NB, lb_pack(epoch, CM_LB_INCL, (uint32_t)k >= abs_from ? c[k] : run + c[k]));
    } else {
      *chain = ((unsigned long long)(b + 1u) << 32) | (unsigned long long)(run + sum);
#pragma unroll
      for (int k = 0; k < RS_SCAN_ROWS; ++k)
        if (r0 + k < n_tiles) st_cg_u64(base + (size_t)k * NB, lb_pack(epoch, CM_LB_INCL, run + c[k]));
    }
  }
}

// Which lanes of the warp hold a different value in bits 0..7 of x: bit j of the result is set iff lane j differs.
// One ballot per bit; a lane whose bit is set complements the ballot, so the OR over bits marks the differing lanes.
// (warp_diff<8> is this; warp_diff<9> takes one ballot more for a digit of up to 511.)
__device__ __forceinline__ uint32_t warp_diff8(uint32_t x) {
  uint32_t t[8];
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    asm volatile(
        "{\n .reg .pred p;\n .reg .b32 y;\n and.b32 y, %1, %2;\n setp.ne.u32 p, y, 0;\n"
        " vote.sync.ballot.b32 %0, p, 0xffffffff;\n @p not.b32 %0, %0;\n}"
        : "=r"(t[b])
        : "r"(x), "r"(1u << b));
  }
  uint32_t a, c;
  asm("lop3.b32 %0, %1, %2, %3, 0xFE;" : "=r"(a) : "r"(t[0]), "r"(t[1]), "r"(t[2]));
  asm("lop3.b32 %0, %1, %2, %3, 0xFE;" : "=r"(c) : "r"(t[3]), "r"(t[4]), "r"(t[5]));
  asm("lop3.b32 %0, %1, %2, %3, 0xFE;" : "=r"(a) : "r"(a), "r"(t[6]), "r"(t[7]));
  return a | c;
}

template <int BITS>
__device__ __forceinline__ uint32_t warp_diff(uint32_t x) {
  if constexpr (BITS == 8) {
    return warp_diff8(x);
  } else {
    static_assert(BITS == 9, "8 or 9 digit bits");
    const uint32_t t8 = warp_diff8(x);
    uint32_t t;
    asm volatile(
        "{\n .reg .pred p;\n .reg .b32 y;\n and.b32 y, %1, %2;\n setp.ne.u32 p, y, 0;\n"
        " vote.sync.ballot.b32 %0, p, 0xffffffff;\n @p not.b32 %0, %0;\n}"
        : "=r"(t)
        : "r"(x), "r"(1u << 8));
    return t8 | t;
  }
}

// The digit a pass ranks. 8-bit passes: bits shift .. shift+7 of the key. Wide top digit (NB = CM_WIDE_BINS, fused-key runs
// sorted frame by frame): the box-grid index bits from shift up, clamped to NB - 1 -- the all-ones key that pads a partial tile
// has 9 set index bits there (the plan takes a wide digit only for 9-bit ones), so it ranks last like digit 255 does.
template <int NB, typename KeyT>
__device__ __forceinline__ uint32_t sort_digit(KeyT k, uint32_t shift, uint32_t idx_mask) {
  if constexpr (NB == CM_RADIX) return (uint32_t)(k >> shift) & (CM_RADIX - 1);
  else return min(((uint32_t)k & idx_mask) >> shift, (uint32_t)NB - 1u);
}

__device__ __forceinline__ uint32_t lanemask_gt() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_gt;" : "=r"(m));
  return m;
}

// Shared memory of one worker CTA. The sorted-tile buffers are double: a CTA ranks and places tile B while the scanners
// are still producing the row that tile A (placed in the other buffer) needs for its scatter -- see the kernel.
// NB: bins of the pass. WIDE_LATER: the FUSED0 pass of a run whose last pass ranks a wide digit (its counters overrun row 3).
template <typename KeyT, int IPT, int NB = CM_RADIX, bool WIDE_LATER = false>
struct SortSmem {
  static constexpr int TILE = RS_THREADS * IPT;
  static constexpr bool AOS = sizeof(KeyT) == 4;
  static constexpr int LATER = 3 * CM_RADIX + (WIDE_LATER ? (int)CM_WIDE_BINS - CM_RADIX : 0);
  unsigned long long k[2][TILE];       // AOS: records (value << 32 | key); else keys
  uint32_t v[2][AOS ? 1 : TILE];       // values of 64-bit keys
  uint32_t hist[RS_WARPS * NB];        // per-warp digit counters, then per-warp first positions
  uint32_t scatter[2][NB];             // global position of sorted-tile position 0 of digit d
  uint32_t scan[NB / 32 + 4];
  uint32_t cnt[NB];                    // RS_EARLY_COUNT: the tile's digit counts, taken before the ranking
  uint32_t later[LATER];               // FUSED0: digit counts of pass ps = 1..3 at (ps - 1) * 256, taken while pass 0 holds the keys
  uint32_t next_tile[2];               // written by thread 0 one iteration ahead (parity-indexed)
};

// FUSED0: pass 0 of a run whose keys were written by K1 at the survivors' slots (VoxelParams::fused_keys): the tile's keys
// are read through the K1 tile records, the value of a key is the slot it was read from.
// SEG: frame-segmented sort (see scanner_cta): tile t is seg_tile[t] -- a range of one frame -- instead of [t TILE, (t+1) TILE).
// FUSED0 && SEG: pass 0 of a fused-key run sorted frame by frame (BoxGrid::seg_sort); K1 counted the pass-0 digits per frame
// and the later passes' digits are counted here per frame (seg_hist), turned into first positions by k_seg_base.
// NB: bins of the pass -- 256, or CM_WIDE_BINS for the wide top digit of a fused-key SEG run (see sort_digit).
template <typename KeyT, int IPT, bool FUSED0 = false, bool SEG = false, int NB = CM_RADIX>
__global__ void __launch_bounds__(RS_THREADS, RS_MIN_CTAS) k_onesweep_pass(const VoxelParams p, const int pass) {
  static_assert(!SEG || sizeof(KeyT) == 4, "segmented keys are 32-bit records");
  static_assert(NB == CM_RADIX || (SEG && !FUSED0 && NB == (int)CM_WIDE_BINS), "a wide digit is the top digit of a SEG run");
  constexpr int TILE = RS_THREADS * IPT;
  constexpr int WARP_ITEMS = 32 * IPT;
  constexpr bool AOS = sizeof(KeyT) == 4;  // (key, value) records of 8 bytes
  constexpr int SCANNERS = NB / RS_SCAN_DIGITS;
  using Smem = SortSmem<KeyT, IPT, NB, FUSED0 && SEG>;
  extern __shared__ __align__(16) unsigned char s_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(s_raw);

  const long long tr0 = clock64();
  const SortInfo si = *p.info;
  if ((uint32_t)pass >= si.num_passes) return;
  if (p.dual_width && ((si.width == 4u) != (sizeof(KeyT) == 4))) return;  // the other key width runs
  if (SEG != (si.seg_sort != 0u)) return;
  const uint32_t M = si.n_keys;
  const uint32_t n_tiles = SEG ? si.n_seg_tiles : (M + TILE - 1) / TILE;
  const uint32_t* const seg_base = SEG ? p.seg_hist + (size_t)pass * CM_RADIX : nullptr;

  const uint32_t tid = threadIdx.x, lane = tid & 31u;
  const uint32_t warp = __shfl_sync(0xFFFFFFFFu, tid >> 5, 0);  // provably warp-uniform
  const uint32_t epoch = *p.epoch_dev + 1u + (uint32_t)pass;
  unsigned long long* const rows = p.lb_sort + NB;  // row -1 lives in front
  uint32_t* const err = &p.ctrl->error;
  // Roles go by ARRIVAL, not by block index: the first RS_SCANNERS CTAs of the pass to start running are the scanners, so
  // the scanners are resident by construction whatever order the hardware dispatches CTAs in and whatever else shares the
  // GPU (several handles sorting on their own streams, MPS). Later arrivals work; a worker publishes its counts before it
  // waits, so the pair cannot deadlock. The same shared-memory hand-over carries the worker's first tile.
  uint32_t* const counter = &p.ctrl->tile_counter[1 + pass];
  if (tid == 0) {
    const uint32_t role = atomicAdd(&p.ctrl->role_counter[pass], 1u);
    sm.next_tile[1] = role;
    if (role >= (uint32_t)SCANNERS) sm.next_tile[0] = atomicAdd(counter, 1u);
  }
  __syncthreads();
  const uint32_t role = sm.next_tile[1];
  if (role < (uint32_t)SCANNERS) {
    __syncthreads();  // every thread has read the role before the scanner reuses the shared memory
    scanner_cta<SEG, NB>(role, rows, n_tiles, epoch, p.hist + pass * CM_RADIX, err, sm.scan, sm.hist, &sm.k[0][0], p.seg_tile, seg_base);
    return;
  }

#define RS_TRACE(t, i, t0) do { if (p.trace && p.trace_pass == (uint32_t)pass && tid == 0) p.trace[(size_t)(t) * 8 + (i)] = (unsigned long long)(clock64() - (t0)); } while (0)
  const bool odd = (pass & 1) != 0;
  const uint32_t shift = (uint32_t)pass * CM_RADIX_BITS;
  const uint32_t lt = lanemask_lt(), gt = lanemask_gt();
  uint32_t* const wh = sm.hist + warp * NB;  // the warp's own counter row
  // wide digit / FUSED0 && SEG: the box-grid index bits of the key (the frame bits above them are not ranked)
  const uint32_t idx_mask = (NB > CM_RADIX || (FUSED0 && SEG)) ? (si.idx_bits >= 32u ? 0xFFFFFFFFu : (1u << si.idx_bits) - 1u) : 0u;
  uint32_t hist_frame = 0xFFFFFFFFu;  // FUSED0 && SEG: the frame sm.later counts for
  // FUSED0 && SEG: sm.later -> the frame's rows of seg_hist (passes 1..), fire-and-forget; cleared for the next frame
  auto flush_later = [&]() {
    if (hist_frame == 0xFFFFFFFFu) return;
    uint32_t* dst = p.seg_hist + (size_t)hist_frame * (CM_SEG_PASSES * CM_RADIX) + CM_RADIX;
    for (uint32_t i = tid; i < (uint32_t)Smem::LATER; i += RS_THREADS) {
      const uint32_t c = sm.later[i];
      if (c) { atomicAdd(dst + i, c); sm.later[i] = 0u; }
    }
  };

  // Tiles are handed out by an atomic counter (forward progress never depends on which CTAs are resident). A CTA works
  // on two tiles at a time, software-pipelined:  front(t1): load, rank, publish counts, place into buffer b1
  //                                              back(t0):  wait for row t0-1 from the scanners, scatter buffer b0
  // so the scanners' latency (poll + chain + store + our poll, ~4-6 thousand cycles) hides behind front(t1) instead of
  // idling a third of the SM's warps as it did when a CTA handled one tile from start to end.
  if (RS_EARLY_COUNT && tid < NB) sm.cnt[tid] = 0;
  if (FUSED0)
    for (uint32_t i = tid; i < (uint32_t)Smem::LATER; i += RS_THREADS) sm.later[i] = 0u;
  uint32_t cur = sm.next_tile[0];
  __syncthreads();  // next_tile[1] (the role) is rewritten below; sm.cnt is cleared
  uint32_t prev = 0xFFFFFFFFu, prev_n = 0;
  uint32_t prev_seg = 0;  // SEG: frame (and first-of-frame bit) of the tile in back()
  uint32_t buf = 0;  // also the parity of the iteration
  long long tr_cur = tr0, tr_prev = tr0;
  uint32_t claimed = 0xFFFFFFFFu;
  while (true) {
    tr_prev = tr_cur;
    tr_cur = clock64();
    const bool have = cur < n_tiles;
    uint32_t n_here = 0;
    uint32_t cur_seg = 0;
    if (have) {
      // ================================= front(cur) ==========================================================
      uint32_t tile_base = cur * TILE;
      if (SEG) {
        const uint4 q = __ldg(reinterpret_cast<const uint4*>(p.seg_tile + cur));
        tile_base = q.x; n_here = q.y; cur_seg = q.z;
      } else {
        n_here = min((uint32_t)TILE, M - tile_base);
      }
      const bool full = n_here == (uint32_t)TILE;
      const uint32_t item0 = warp * WARP_ITEMS + lane;  // tile-local index of item 0 of this thread; item i = item0 + 32 i
      // ---- load keys and values (warp-striped, coalesced). Slots past the end of a partial (last) tile get the
      // all-ones key: digit 255 in every pass, and -- being the last items of the tile -- ranked after every real key
      // of that digit, so they land at sorted-tile positions >= n_here and are simply not written back.
      KeyT key[IPT];
      uint32_t val[IPT];
      if (FUSED0) {
        // Dense position d of the merged cropped cloud -> slot: K1 tile e holds positions [dense0_e, dense0_e + count_e) at slots
        // slot0_e + (d - dense0_e). Lane l of every warp holds the record of K1 tile first + l (a radix tile spans a handful
        // of K1 tiles); the tile of a position is the last one whose dense0 does not exceed it.
        if (SEG && (cur_seg & ~CM_SEG_FIRST) != hist_frame) {  // CTA-uniform; the last tile's increments are done
          flush_later();
          hist_frame = cur_seg & ~CM_SEG_FIRST;
          __syncthreads();
        }
        const uint32_t k1_first = p.first_k1[cur];
        const uint32_t e = k1_first + lane;
        uint32_t e_dense = 0xFFFFFFFFu, e_slot = 0u, e_end = 0xFFFFFFFFu;
        if (e < p.n_k1_tiles) {
          const uint4 q = __ldg(reinterpret_cast<const uint4*>(p.tile_rec + e));
          e_dense = q.w; e_slot = q.y; e_end = q.w + q.x;
        }
        const uint32_t last_end = __shfl_sync(0xFFFFFFFFu, e_end, 31);
        const bool covered = last_end >= tile_base + n_here;  // (entries past the last K1 tile count as covering)
        const uint32_t w0 = tile_base + warp * WARP_ITEMS;
        uint32_t kk = (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, e_dense <= w0));
        kk = kk ? kk - 1u : 0u;
        const uint32_t* __restrict__ tdense = reinterpret_cast<const uint32_t*>(p.tile_rec);
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
          const uint32_t d = tile_base + item0 + 32 * i;
          uint32_t slot;
          if (covered) {
            bool adv;
            do {  // positions grow with i, so the entry index only ever moves forward
              const uint32_t nd = __shfl_sync(0xFFFFFFFFu, e_dense, (kk + 1u) & 31u);
              adv = kk < 31u && nd <= d;
              kk += adv ? 1u : 0u;
            } while (__any_sync(0xFFFFFFFFu, adv));
            slot = __shfl_sync(0xFFFFFFFFu, e_slot, kk) + (d - __shfl_sync(0xFFFFFFFFu, e_dense, kk));
          } else {
            // a radix tile that spans more than 32 K1 tiles (a crop that keeps a few percent): binary search in global memory
            uint32_t lo = k1_first, hi = p.n_k1_tiles - 1u;
            while (lo < hi) {
              const uint32_t mid = (lo + hi + 1u) >> 1;
              if (tdense[mid * 4u + 3u] <= d) lo = mid; else hi = mid - 1u;
            }
            slot = tdense[lo * 4u + 1u] + (d - tdense[lo * 4u + 3u]);
          }
          const bool in = SEG ? item0 + 32 * i < n_here : d < M;
          key[i] = in ? (KeyT)p.surv_key[slot] : ~(KeyT)0;
          val[i] = in ? slot : 0u;
        }
        // K1 counted the digits of pass 0 only; the later passes' histograms are taken here, where every key passes once
        if (SEG) {  // the frame's counts; the last pass ranks a wide digit when the plan says so
          const uint32_t wide_pass = p.box.top_bins > CM_RADIX ? si.num_passes - 1u : 0u;
#pragma unroll
          for (int i = 0; i < IPT; ++i) {
            if (item0 + 32 * i < n_here) {
#pragma unroll
              for (uint32_t ps = 1; ps < 3; ++ps)
                if (ps < si.num_passes) {
                  const uint32_t dg = ps == wide_pass ? sort_digit<(int)CM_WIDE_BINS>((uint32_t)key[i], ps * CM_RADIX_BITS, idx_mask)
                                                      : sort_digit<CM_RADIX>((uint32_t)key[i], ps * CM_RADIX_BITS, 0u);
                  atomicAdd(&sm.later[(ps - 1) * CM_RADIX + dg], 1u);
                }
            }
          }
        } else {
#pragma unroll
          for (int i = 0; i < IPT; ++i) {
            if (tile_base + item0 + 32 * i < M) {
#pragma unroll
              for (uint32_t ps = 1; ps < 4; ++ps)
                if (ps < si.num_passes) atomicAdd(&sm.later[(ps - 1) * CM_RADIX + (((uint32_t)key[i] >> (ps * CM_RADIX_BITS)) & (CM_RADIX - 1))], 1u);
            }
          }
        }
      } else if (AOS) {
        const uint2* __restrict__ in = reinterpret_cast<const uint2*>(odd ? p.keys_b : p.keys_a) + tile_base + item0;
        if (full) {
#pragma unroll
          for (int i = 0; i < IPT; ++i) {
            const uint2 r = in[32 * i];
            key[i] = (KeyT)r.x;
            val[i] = r.y;
          }
        } else {
#pragma unroll
          for (int i = 0; i < IPT; ++i) {
            uint2 r = make_uint2(0xFFFFFFFFu, 0u);
            if (item0 + 32 * i < n_here) r = in[32 * i];
            key[i] = (KeyT)r.x;
            val[i] = r.y;
          }
        }
      } else {
        const KeyT* __restrict__ in_keys = reinterpret_cast<const KeyT*>(odd ? p.keys_b : p.keys_a) + tile_base + item0;
        const uint32_t* __restrict__ in_vals = (odd ? p.vals_b : p.vals_a) + tile_base + item0;
        if (full) {
#pragma unroll
          for (int i = 0; i < IPT; ++i) key[i] = in_keys[32 * i];
#pragma unroll
          for (int i = 0; i < IPT; ++i) val[i] = in_vals[32 * i];
        } else {
#pragma unroll
          for (int i = 0; i < IPT; ++i) key[i] = (item0 + 32 * i < n_here) ? in_keys[32 * i] : ~(KeyT)0;
#pragma unroll
          for (int i = 0; i < IPT; ++i) val[i] = (item0 + 32 * i < n_here) ? in_vals[32 * i] : 0u;
        }
      }
#pragma unroll
      for (int k = 0; k < NB / 32; ++k) wh[lane + 32 * k] = 0;
      __syncwarp();
      RS_TRACE(cur, 0, tr_cur);
      if (RS_EARLY_COUNT) {
        // The tile's digit counts go out before the (long) ranking: one hardware-aggregated shared-memory increment per
        // key (ATOMS.POPC.INC). The later a tile publishes, the longer every tile after it waits for its row.
#pragma unroll
        for (int i = 0; i < IPT; ++i) atomicAdd(&sm.cnt[sort_digit<NB>(key[i], shift, idx_mask)], 1u);
        __syncthreads();
        if (RS_THREADS == NB || tid < NB) {
          const uint32_t c = sm.cnt[tid];
          sm.cnt[tid] = 0;  // for the next tile (no increments can follow in this iteration)
          const uint32_t real = (tid == NB - 1) ? c - ((uint32_t)TILE - n_here) : c;
          st_relaxed_u64(rows + (size_t)cur * NB + tid, lb_pack(epoch, CM_LB_AGG, real));
        }
      }

      // ---- stable rank of every key among the keys of its digit inside the warp ------------------------------------
      // peers = lanes holding the same digit (ballot match, constant time; __match_any_sync costs one round per
      // distinct value). Every lane reads the digit's counter; the highest peer lane writes it back advanced by the
      // peer count. Shared-memory accesses of one warp are performed in program order; __syncwarp keeps the compiler
      // from reordering them.
      uint32_t rank[IPT];
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        uint32_t ks, diff;
        if constexpr (NB == CM_RADIX) {
          ks = (uint32_t)(key[i] >> shift);
          diff = warp_diff<8>(ks);
          ks &= CM_RADIX - 1;
        } else {
          ks = sort_digit<NB>(key[i], shift, idx_mask);
          diff = warp_diff<9>(ks);
        }
        const uint32_t below = (uint32_t)__popc(~diff & lt);
        volatile uint32_t* c = wh + ks;
        const uint32_t r = *c + below;
        rank[i] = r;
        if ((~diff & gt) == 0u) *c = r + 1u;
        __syncwarp();
      }
      __syncthreads();
      RS_TRACE(cur, 1, tr_cur);

      // ---- per digit (one per thread): tile count -> published; prefix over digits and warps -> first positions -----
      {
        const bool dt = RS_THREADS == NB || tid < NB;  // digit threads
        uint32_t wc[RS_WARPS];
        uint32_t cnt = 0;
        if (dt) {
#pragma unroll
          for (int w = 0; w < RS_WARPS; ++w) {
            wc[w] = sm.hist[w * NB + tid];
            cnt += wc[w];
          }
          if (!RS_EARLY_COUNT) {
            const uint32_t real = (tid == NB - 1) ? cnt - ((uint32_t)TILE - n_here) : cnt;
            st_relaxed_u64(rows + (size_t)cur * NB + tid, lb_pack(epoch, CM_LB_AGG, real));
          }
        }
        RS_TRACE(cur, 2, tr_cur);
        uint32_t tot;
        const uint32_t bin_start = block_excl_scan<NB>(cnt, sm.scan, &tot);
        if (dt) {
          uint32_t run = bin_start;
#pragma unroll
          for (int w = 0; w < RS_WARPS; ++w) {
            sm.hist[w * NB + tid] = run;
            run += wc[w];
          }
          sm.scatter[buf][tid] = 0u - bin_start;  // completed in back() once the scanners have delivered the row
        }
      }
      __syncthreads();
      RS_TRACE(cur, 3, tr_cur);

      // ---- keys and values into sorted-tile order in shared memory -------------------------------------------------
#pragma unroll
      for (int i = 0; i < IPT; ++i) {
        const uint32_t pos = wh[sort_digit<NB>(key[i], shift, idx_mask)] + rank[i];
        if (AOS) {
          sm.k[buf][pos] = ((unsigned long long)val[i] << 32) | (unsigned long long)key[i];
        } else {
          sm.k[buf][pos] = (unsigned long long)key[i];
          sm.v[buf][pos] = val[i];
        }
      }
      RS_TRACE(cur, 4, tr_cur);
    }
    if (prev != 0xFFFFFFFFu) {
      // ================================= back(prev) ===========================================================
      const uint32_t pb = buf ^ 1u;
      RS_TRACE(prev, 7, tr_prev);
      // ---- one row from the scanners: where this tile's keys of digit d start in the output ----------------------
      if (RS_THREADS == NB || tid < NB) {
        uint32_t first;
        if (SEG && (prev_seg & CM_SEG_FIRST))  // first tile of its frame: the frame's own first positions, nobody to wait for
          first = __ldg(seg_base + (size_t)(prev_seg & ~CM_SEG_FIRST) * (CM_SEG_PASSES * CM_RADIX) + tid);
        else
          first = lb_wait_inclusive(rows + ((long long)prev - 1) * NB + tid, epoch, err);
        sm.scatter[pb][tid] += first;  // modulo 2^32
      }
      __syncthreads();
      RS_TRACE(prev, 5, tr_prev);
      // Claim the next tile now, not earlier: a tile claimed long before its front() runs holds back the published
      // frontier for every later tile. The result is only needed after the scatter below, so its latency is hidden.
      if (tid == 0 && have) claimed = atomicAdd(counter, 1u);
      // ---- scatter: consecutive threads write consecutive addresses inside each digit's run -----------------------
      // (two copies of the loop: the one for full tiles carries no bounds checks, so its shared-memory loads batch up)
      const bool pfull = prev_n == (uint32_t)TILE;
      const unsigned long long* sk = sm.k[pb];
      const uint32_t* ssc = sm.scatter[pb];
      if (AOS) {
        unsigned long long* __restrict__ out = reinterpret_cast<unsigned long long*>(odd ? p.keys_a : p.keys_b);
        if (pfull) {
          unsigned long long r[IPT];
#pragma unroll
          for (int j = 0; j < IPT; ++j) r[j] = sk[j * RS_THREADS + tid];
#pragma unroll
          for (int j = 0; j < IPT; ++j) {
            const uint32_t dg = sort_digit<NB>((uint32_t)r[j], shift, idx_mask);
            out[ssc[dg] + (j * RS_THREADS + tid)] = r[j];
          }
        } else {
          for (uint32_t pos = tid; pos < prev_n; pos += RS_THREADS) {
            const unsigned long long r = sk[pos];
            const uint32_t dg = sort_digit<NB>((uint32_t)r, shift, idx_mask);
            out[ssc[dg] + pos] = r;
          }
        }
      } else {
        KeyT* __restrict__ out_keys = reinterpret_cast<KeyT*>(odd ? p.keys_a : p.keys_b);
        uint32_t* __restrict__ out_vals = odd ? p.vals_a : p.vals_b;
        const uint32_t* sv = sm.v[pb];
        if (pfull) {
#pragma unroll
          for (int j0 = 0; j0 < IPT; j0 += 4) {
            unsigned long long kk[4];
            uint32_t vv[4];
#pragma unroll
            for (int j = 0; j < 4 && j0 + j < IPT; ++j) {
              kk[j] = sk[(j0 + j) * RS_THREADS + tid];
              vv[j] = sv[(j0 + j) * RS_THREADS + tid];
            }
#pragma unroll
            for (int j = 0; j < 4 && j0 + j < IPT; ++j) {
              const uint32_t dg = (uint32_t)(kk[j] >> shift) & (CM_RADIX - 1);
              const uint32_t dst = ssc[dg] + ((j0 + j) * RS_THREADS + tid);
              out_keys[dst] = (KeyT)kk[j];
              out_vals[dst] = vv[j];
            }
          }
        } else {
          for (uint32_t pos = tid; pos < prev_n; pos += RS_THREADS) {
            const unsigned long long kk = sk[pos];
            const uint32_t dg = (uint32_t)(kk >> shift) & (CM_RADIX - 1);
            const uint32_t dst = ssc[dg] + pos;
            out_keys[dst] = (KeyT)kk;
            out_vals[dst] = sv[pos];
          }
        }
      }
      RS_TRACE(prev, 6, tr_prev);
    } else if (tid == 0 && have) {
      claimed = atomicAdd(counter, 1u);  // first iteration: nothing to scatter yet
    }
    if (!have) break;
    if (tid == 0) sm.next_tile[buf ^ 1u] = claimed;
    prev = cur;
    prev_n = n_here;
    prev_seg = cur_seg;
    buf ^= 1u;
    // Orders this iteration's shared-memory reads (placement reads of the counter rows, scatter reads of the other
    // buffer) before the next iteration's writes, and makes next_tile (written long ago by thread 0) visible.
    __syncthreads();
    cur = sm.next_tile[buf];
  }
  if (FUSED0) {  // this CTA's share of the histograms of passes 1.. (a persistent CTA flushes once, SEG: per frame)
    __syncthreads();
    if (SEG) {
      flush_later();
    } else {
      for (uint32_t i = tid; i < 3u * CM_RADIX; i += RS_THREADS) {
        const uint32_t c = sm.later[i];
        if (c && (i >> 8) + 1u < si.num_passes) atomicAdd(p.hist + CM_RADIX + i, c);
      }
    }
  }
}

// 32-bit keys leave the sort as 8-byte (key, value) records; callers that want two plain arrays get them from here.
__global__ void __launch_bounds__(256) k_split_records(const uint2* __restrict__ rec, uint32_t* __restrict__ keys,
                                                       uint32_t* __restrict__ vals, const uint32_t* n_ptr, const BoxGrid box,
                                                       const GridDev* __restrict__ grid, const SortInfo* info, uint32_t n_frames) {
  const uint32_t n = *n_ptr;
  const uint32_t idx_bits = info ? info->idx_bits : 0u;
  for (uint32_t i = blockIdx.x * 256u + threadIdx.x; i < n; i += gridDim.x * 256u) {
    const uint2 r = rec[i];
    uint32_t key = r.x;
    if (grid) {  // box-grid index -> PCL's idx on the frame's own grid
      const uint32_t f = idx_bits < 32u ? key >> idx_bits : 0u;
      const uint32_t b = idx_bits < 32u ? key & ((1u << idx_bits) - 1u) : key;
      const uint32_t k2 = b / box.mul2, r2 = b - k2 * box.mul2, k1 = r2 / box.mul1, k0 = r2 - k1 * box.mul1;
      const GridDev* g = grid + (f < n_frames ? f : 0u);
      const long long c0 = (long long)k0 + box.min_b[0] - g->min_b[0], c1 = (long long)k1 + box.min_b[1] - g->min_b[1],
                      c2 = (long long)k2 + box.min_b[2] - g->min_b[2];
      key = (idx_bits < 32u ? f << idx_bits : 0u) | (uint32_t)(c0 + c1 * (long long)g->mul1 + c2 * (long long)g->mul2);
    }
    keys[i] = key;
    vals[i] = r.y;
  }
}

}  // namespace

// Two tile sizes per key width. A single frame (a few hundred thousand keys) cut into 4608-key tiles would occupy a third
// of the SMs with one long tile each; 1536-key tiles spread it over the chip and shorten the critical path of a pass.
constexpr int RS_IPT_SMALL = 4;
constexpr uint32_t RS_SMALL_LIMIT = 148u * 2u * RS_THREADS * RS_IPT32;  // up to ~1.4 M keys: the small tile

static bool sort_uses_small_tile(uint32_t max_points) { return max_points <= RS_SMALL_LIMIT; }

uint32_t sort_tile_items(uint32_t key_bytes, uint32_t max_points) {
  if (sort_uses_small_tile(max_points)) return RS_THREADS * RS_IPT_SMALL;
  return key_bytes == 4 ? RS_THREADS * SortCfg<uint32_t>::IPT : RS_THREADS * SortCfg<unsigned long long>::IPT;
}

// rows of look-back words a workspace of `capacity` points needs (+1 for row -1, +1 spare)
// (a frame-segmented sort needs one more row per frame, and a wide top digit rows of CM_WIDE_BINS words: see ws_alloc)
size_t sort_lookback_rows(uint32_t capacity) {
  const uint32_t small_part = std::min(capacity, RS_SMALL_LIMIT);
  const size_t rows_small = small_part / (RS_THREADS * RS_IPT_SMALL) + 1;
  const size_t rows_big = capacity / (RS_THREADS * std::min<int>(SortCfg<uint32_t>::IPT, SortCfg<unsigned long long>::IPT)) + 1;
  return std::max(rows_small, rows_big) + 2;
}

namespace {
template <typename KeyT, int IPT, bool FUSED0 = false, bool SEG = false, int NB = CM_RADIX>
struct PassLaunch {
  using Smem = SortSmem<KeyT, IPT, NB, FUSED0 && SEG>;
  static constexpr uint32_t SCANNERS = NB / RS_SCAN_DIGITS;
  static inline int ctas_per_sm = 0;
  static cudaError_t configure() {
    cudaError_t e = cudaFuncSetAttribute(k_onesweep_pass<KeyT, IPT, FUSED0, SEG, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)sizeof(Smem));
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, k_onesweep_pass<KeyT, IPT, FUSED0, SEG, NB>, RS_THREADS,
                                                         sizeof(Smem));
  }
  static cudaError_t launch(const VoxelParams& p, int pass, int sms, cudaStream_t stream) {
    const uint32_t tile = RS_THREADS * IPT;
    const uint32_t tiles = (p.max_points + tile - 1) / tile + (SEG ? p.n_frames : 0u);  // SEG: a partial tile per frame
    if (tiles == 0) return cudaSuccess;
    // persistent workers: at most what the device holds at once (tiles are handed out by an atomic counter)
    const uint32_t workers = std::min<uint32_t>(tiles, (uint32_t)(sms * std::max(1, ctas_per_sm)) - SCANNERS);
    k_onesweep_pass<KeyT, IPT, FUSED0, SEG, NB><<<workers + SCANNERS, RS_THREADS, sizeof(Smem), stream>>>(p, pass);
    return cudaGetLastError();
  }
};
bool g_sort_configured = false;
}  // namespace

cudaError_t configure_sort_kernels() {
  if (g_sort_configured) return cudaSuccess;
  cudaError_t e = PassLaunch<uint32_t, SortCfg<uint32_t>::IPT>::configure();
  if (e == cudaSuccess) e = PassLaunch<unsigned long long, SortCfg<unsigned long long>::IPT>::configure();
  if (e == cudaSuccess) e = PassLaunch<uint32_t, RS_IPT_SMALL>::configure();
  if (e == cudaSuccess) e = PassLaunch<unsigned long long, RS_IPT_SMALL>::configure();
  if (e == cudaSuccess) e = PassLaunch<uint32_t, SortCfg<uint32_t>::IPT, true>::configure();
  if (e == cudaSuccess) e = PassLaunch<uint32_t, RS_IPT_SMALL, true>::configure();
  if (e == cudaSuccess) e = PassLaunch<uint32_t, SortCfg<uint32_t>::IPT, false, true>::configure();
  if (e == cudaSuccess) e = PassLaunch<uint32_t, RS_IPT_SMALL, false, true>::configure();
  if (e == cudaSuccess) e = PassLaunch<uint32_t, SortCfg<uint32_t>::IPT, true, true>::configure();
  if (e == cudaSuccess) e = PassLaunch<uint32_t, RS_IPT_SMALL, true, true>::configure();
  if (e == cudaSuccess) e = PassLaunch<uint32_t, SortCfg<uint32_t>::IPT, false, true, CM_WIDE_BINS>::configure();
  if (e == cudaSuccess) e = PassLaunch<uint32_t, RS_IPT_SMALL, false, true, CM_WIDE_BINS>::configure();
  if (e != cudaSuccess) return e;
  if (getenv("CM_DEBUG"))
    fprintf(stderr, "[cm] sort pass CTAs per SM: %d / %d (32 / 64-bit keys), small tile %d / %d, wide top digit %d / %d\n",
            PassLaunch<uint32_t, SortCfg<uint32_t>::IPT>::ctas_per_sm,
            PassLaunch<unsigned long long, SortCfg<unsigned long long>::IPT>::ctas_per_sm,
            PassLaunch<uint32_t, RS_IPT_SMALL>::ctas_per_sm, PassLaunch<unsigned long long, RS_IPT_SMALL>::ctas_per_sm,
            PassLaunch<uint32_t, SortCfg<uint32_t>::IPT, false, true, CM_WIDE_BINS>::ctas_per_sm,
            PassLaunch<uint32_t, RS_IPT_SMALL, false, true, CM_WIDE_BINS>::ctas_per_sm);
  g_sort_configured = true;
  return cudaSuccess;
}

cudaError_t launch_sort_pass(const VoxelParams& p, int pass, cudaStream_t stream) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const bool small = sort_uses_small_tile(p.max_points);
  if (p.fused_keys && p.box.seg_sort) {  // frame by frame, 32-bit keys; the last pass may rank a wide digit
    constexpr int I = SortCfg<uint32_t>::IPT;
    if (pass == 0)
      return small ? PassLaunch<uint32_t, RS_IPT_SMALL, true, true>::launch(p, pass, sms, stream)
                   : PassLaunch<uint32_t, I, true, true>::launch(p, pass, sms, stream);
    if ((uint32_t)pass + 1u == p.box.n_pass && p.box.top_bins > CM_RADIX)
      return small ? PassLaunch<uint32_t, RS_IPT_SMALL, false, true, CM_WIDE_BINS>::launch(p, pass, sms, stream)
                   : PassLaunch<uint32_t, I, false, true, CM_WIDE_BINS>::launch(p, pass, sms, stream);
    return small ? PassLaunch<uint32_t, RS_IPT_SMALL, false, true>::launch(p, pass, sms, stream)
                 : PassLaunch<uint32_t, I, false, true>::launch(p, pass, sms, stream);
  }
  if (p.fused_keys && pass == 0)  // 32-bit keys by construction
    return small ? PassLaunch<uint32_t, RS_IPT_SMALL, true>::launch(p, pass, sms, stream)
                 : PassLaunch<uint32_t, SortCfg<uint32_t>::IPT, true>::launch(p, pass, sms, stream);
  if (p.key_bytes == 4 && p.segmented)
    return small ? PassLaunch<uint32_t, RS_IPT_SMALL, false, true>::launch(p, pass, sms, stream)
                 : PassLaunch<uint32_t, SortCfg<uint32_t>::IPT, false, true>::launch(p, pass, sms, stream);
  if (p.key_bytes == 4)
    return small ? PassLaunch<uint32_t, RS_IPT_SMALL>::launch(p, pass, sms, stream)
                 : PassLaunch<uint32_t, SortCfg<uint32_t>::IPT>::launch(p, pass, sms, stream);
  return small ? PassLaunch<unsigned long long, RS_IPT_SMALL>::launch(p, pass, sms, stream)
               : PassLaunch<unsigned long long, SortCfg<unsigned long long>::IPT>::launch(p, pass, sms, stream);
}

cudaError_t launch_split_records(const void* records, uint32_t* keys, uint32_t* vals, const uint32_t* n_ptr,
                                 uint32_t max_points, cudaStream_t stream, const VoxelParams* remap) {
  if (max_points == 0) return cudaSuccess;
  const uint32_t blocks = std::min<uint32_t>((max_points + 255u) / 256u, 148u * 8u);
  k_split_records<<<blocks, 256, 0, stream>>>(reinterpret_cast<const uint2*>(records), keys, vals, n_ptr,
                                              remap ? remap->box : BoxGrid{}, remap ? remap->grid : nullptr,
                                              remap ? remap->info : nullptr, remap ? remap->n_frames : 0u);
  return cudaGetLastError();
}

}  // namespace cm
