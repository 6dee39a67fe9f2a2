// cm_api.cu -- host side of the C ABI declared in include/cloud_merger_gpu.h.
//
// Owns every device allocation (made once, at creation / first use -- no per-frame cudaMalloc), the per-sensor copy
// streams, the frame slots of the host path and the launch sequence of a run:
//     memset(control block) -> K1 transform_crop -> grid_setup -> key_hist -> P x onesweep pass -> centroid
// There is no CPU implementation behind any entry point: without a CUDA device cm_create fails.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <sched.h>
#include <nccl.h>  // types only: the library is loaded at run time (cm_giant_*), see NcclApi

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <mutex>
#include <new>
#include <random>
#include <string>
#include <type_traits>
#include <unordered_map>
#include <vector>

#include "../../include/cloud_merger_gpu.h"
#include "cm_kernels.h"

using namespace cm;

namespace {

constexpr size_t kAlign = 256;
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Owners of the CUDA resources: a set-up that fails part-way leaves nothing behind once its struct is reset or destroyed.
struct CudaFree { void operator()(void* p) const { cudaFree(p); } };
struct CudaFreeHost { void operator()(void* p) const { cudaFreeHost(p); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct GraphExecDestroy { void operator()(cudaGraphExec_t g) const { cudaGraphExecDestroy(g); } };
template <typename T> using DevPtr = std::unique_ptr<T, CudaFree>;
template <typename T> using HostPtr = std::unique_ptr<T, CudaFreeHost>;  // default and mapped page-locked memory
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;
using GraphExec = std::unique_ptr<std::remove_pointer_t<cudaGraphExec_t>, GraphExecDestroy>;

struct MetaLayout {
  size_t off_ctrl, off_acc, off_hist, zero_bytes, off_info, off_fstart, off_segstart, off_grid, total;
  void build(uint32_t frames, uint32_t segs) {
    off_ctrl = 0;
    off_acc = align_up(sizeof(Ctrl), 64);
    off_hist = align_up(off_acc + sizeof(FrameAcc) * frames, 64);
    zero_bytes = off_hist + sizeof(uint32_t) * CM_MAX_SORT_PASSES * CM_RADIX;
    off_info = align_up(zero_bytes, 64);
    off_fstart = align_up(off_info + sizeof(SortInfo), 64);
    off_segstart = align_up(off_fstart + sizeof(uint32_t) * (frames + 1), 64);
    off_grid = align_up(off_segstart + sizeof(uint32_t) * segs, 64);
    total = align_up(off_grid + sizeof(GridDev) * frames, 256);
  }
};

enum StageEv { EV_START = 0, EV_K1, EV_GRID, EV_KEY, EV_SORT, EV_CENT, EV_SORT0 /* after radix pass 0 */, EV_COUNT };

struct Workspace {
  bool ready = false;
  uint32_t cap_points = 0, cap_frames = 0, cap_segs = 0;
  uint32_t plan_idx_bits = 0, plan_total_bits = 0;  // key plan of the last unbounded run (fetched from the device)
  uint32_t plan_error = 0;                          // Ctrl.error when that plan was fetched (k_grid_setup's verdict)
  int out_step = 16;
  MetaLayout ml{};
  DevPtr<uint8_t> meta;
  HostPtr<uint8_t> report;  // pinned host mirror of meta
  DevPtr<SegDev> segs;
  std::vector<SegDev> segs_host;  // what is currently uploaded
  DevPtr<uint32_t> tile_seg;
  std::vector<uint32_t> tile_seg_host;
  DevPtr<OrientedBoxDev> obox;               // CropBox stages (allocated on first use)
  std::vector<OrientedBoxDev> obox_host;     // what is currently uploaded
  DevPtr<float4> surv_xyzi;
  DevPtr<uint32_t> surv_src;
  DevPtr<uint32_t> surv_key;             // box-grid voxel keys written by K1 (fused-key runs)
  DevPtr<uint32_t> first_k1;             // [sort tiles] K1 tile holding the first key of every radix tile
  DevPtr<SegTile> seg_tile;              // frame-segmented sort (batches of several frames): [sort tiles + frames]
  DevPtr<uint32_t> seg_hist;             //   [frames][CM_SEG_PASSES][256]
  DevPtr<uint32_t> seg_frame_tile0;      //   [frames + 1]
  DevPtr<uint2> seg_cent_range;          //   [centroid tiles]
  bool timed_pass0 = false;              // last run: an event was recorded after radix pass 0 (profiling, host-planned key width)
  bool segmented = false;                // last run: the frame-segmented kernels were enqueued (SortInfo says whether they ran)
  bool fused_keys = false;               // last run: K1 produced the keys
  BoxGrid box{};
  DevPtr<unsigned long long> keys_a, keys_b;
  DevPtr<uint32_t> vals_a, vals_b;
  DevPtr<TileRec> tile_rec;             // [lb_k1_n] K1 tile records
  DevPtr<unsigned long long> cent_status;  // [lb_cent_n] look-back words of the voxel compaction
  DevPtr<unsigned long long> lb_sort;
  DevPtr<uint32_t> epoch_dev;           // run epoch of the look-back words (device-resident, see VoxelParams)
  size_t lb_k1_n = 0, lb_sort_n = 0, lb_cent_n = 0;
  DevPtr<float4> dense_xyzi;            // dense merged cloud, allocated and filled on request only
  DevPtr<uint32_t> dense_src;
  DevPtr<uint32_t> dense_slot;
  bool dense_valid = false;
  uint32_t n_k1_tiles = 0;
  DevPtr<uint8_t> out_xyzi;
  DevPtr<uint32_t> out_count;
  DevPtr<unsigned long long> out_idx;
  DevPtr<unsigned long long> trace_k1;  // debug traces (CM_TRACE=1): 8 stamps per tile
  DevPtr<unsigned long long> trace_sort;
  size_t trace_k1_n = 0, trace_sort_n = 0;
  Event ev[EV_COUNT];
  // description of the last run
  bool has_run = false, report_valid = false, profiled = false;
  uint32_t n_frames = 0, n_segs = 0;
  int64_t points_in = 0;
  uint32_t key_bytes = 8, max_passes = 8;
  const float4* voxel_pts = nullptr;  // points the voxel stage read (survivors or the caller's cloud)
  bool ran_k1 = false, ran_voxel = false;
  bool dual_width = false; // last run: both key widths were enqueued, the device picked one (key_bytes comes with the report)
  bool capturing = false;  // the run is being captured into a graph: its timing events are recorded around the graph launch instead
  int64_t launches = 0;
  cudaStream_t stream = nullptr;
};

struct SensorState {
  bool submitted = false;
  uint8_t* dev = nullptr;  // where this submission's records sit in the slot's raw buffer
  int64_t n_points = 0;
  cm_layout_t layout{};
  uint64_t stamp = 0;
  Event copied;
};

struct Slot {
  Workspace ws;
  DevPtr<uint8_t> raw_dev;        // one region per sensor (single submissions, carried-over clouds)
  HostPtr<uint8_t> raw_pinned;
  // cm_submit_clouds_pinned: host-adjacent clouds travel as one copy into this bump-allocated arena, so a coalesced run
  // never shares bytes with a sensor's own region or with another run; reset when the slot's frame has been merged
  DevPtr<uint8_t> arena_dev;
  size_t arena_bytes = 0, arena_used = 0;
  // page-locked, device-mapped mirrors of the frame's voxel outputs: the last kernel of the frame (k_export_voxels) writes
  // them over PCIe, sized on the device, so cm_wait_frame needs ONE synchronisation and no copy of its own
  HostPtr<uint8_t> exp_xyzi;
  HostPtr<uint32_t> exp_count;
  HostPtr<unsigned long long> exp_idx;
  uint32_t exp_cap = 0;
  std::vector<SensorState> sensor;
  Stream stream;
  Event done;
  int64_t ticket = -1;
  bool busy = false;
  uint64_t used_mask = 0, stamp = 0;
  // The launch sequence of a frame, captured once per configuration and replayed as a CUDA graph: a frame of the host
  // path is ~12 stream operations on half a million points, and enqueueing them one by one costs more host time than
  // the GPU needs to run them. graph_seen: configuration of the previous frame (run the plain way, which also uploads
  // the segment table); graph_key: configuration the instantiated graph belongs to.
  GraphExec graph;
  std::string graph_key, graph_seen;
};

}  // namespace

struct cm_handle_s {
  cm_config_t cfg{};
  int device = 0;
  std::mutex mu;
  std::string last_error;
  // configuration
  float mats_host[CM_MAX_SENSORS * 12];
  CropDev crop{};
  OrientedBoxDev obox[CM_MAX_CROP_BOXES]{};  // cm_set_crop_boxes
  int n_obox = 0;
  float leaf[3] = {0.1f, 0.1f, 0.1f};
  float inv_leaf[3] = {10.f, 10.f, 10.f};
  uint32_t min_points = 2;
  uint32_t downsample_all = 1;
  int overflow_mode = 0;
  bool profiling = false;
  bool have_bounds = false;   // externally supplied bounding box for cm_dev_voxelgrid (partitioned giant cloud)
  uint32_t epoch_start = 0;   // first run epoch of every workspace's look-back words (CM_EPOCH_START, read by cm_create)
  float bounds_min[3] = {0, 0, 0}, bounds_max[3] = {0, 0, 0};
  // run bookkeeping
  uint32_t run_counter = 0;
  Workspace batch;          // device-resident batch path
  Workspace* last = nullptr;  // workspace of the most recent run
  std::vector<cm_frame_info_t> frame_info;
  cm_stats_t stats{};
  float stage_ms[EV_COUNT]{};
  // zone slicing (allocated on first use)
  ZoneSet zones{};
  struct ZoneWs {
    size_t cap_points = 0, cap_out = 0;
    DevPtr<unsigned short> mask;
    DevPtr<uint32_t> tile_count, tile_offset, zone_begin, overflow;
    DevPtr<uint32_t> zone_total;  // [CM_MAX_ZONES] + the scan ticket behind it
    DevPtr<float4> out_xyzi;
    DevPtr<uint32_t> out_src;
    HostPtr<uint32_t> report;     // pinned: zone_begin[CM_MAX_ZONES + 1] + overflow + a radius run's device error word
    cudaStream_t stream = nullptr;
    bool ran = false;
    int64_t launches = 0;
    ZoneParams last{};           // the last split, so that its scatter can be repeated after the outputs grew
    int n_zones_run = 0;         // zones of the last split (1 for a radius outlier removal)
    bool ror_run = false;        // the last split compacted a radius outlier removal: report[CM_MAX_ZONES + 2] holds the
                                 // error word of its count kernel (the 2^14-cell bound of the cell margin)
  } zw;
  // the outlier removals' cell table: first sorted position of every cell key (allocated on first use, grows)
  DevPtr<uint32_t> cell_table;
  size_t cell_table_cap = 0;
  // host-buffer forms: the caller's cloud uploaded (allocated on first use, grows)
  DevPtr<float4> stage;
  size_t stage_cap = 0;
  // statistical outlier removal (allocated on first use, grows)
  struct SorWs {
    size_t cap = 0;
    DevPtr<float4> sorted_pts;     // [cap] the points in sorted key order
    DevPtr<float> dist;            // [cap] mean distance per input point
    DevPtr<SorStats> stats;        // [CM_MAX_ZONES]
    HostPtr<SorStats> stats_host;  // pinned mirror, copied at the end of every run
    Event ev[3];                   // profiling: before the search, after it, after the sums
    cudaStream_t stream = nullptr;
    bool ran = false, profiled = false;
    int n_clouds = 0;
    int64_t n_points = 0;
    uint32_t n_valid[CM_MAX_ZONES] = {};
    uint32_t too_few = 0;
  } sw;
  // RANSAC ground plane (allocated on first use): one batch of draws and its scores, device + pinned mirrors
  struct PlaneWs {
    size_t cap_draws = 0;
    DevPtr<int32_t> samples_dev;  // [cap_draws][3]
    DevPtr<int32_t> counts_dev;   // [cap_draws] counts, then [cap_draws] good flags
    DevPtr<float4> models_dev;    // [cap_draws]
    DevPtr<float> acc_dev;        // [10] running sums + count
    HostPtr<int32_t> samples_pin;
    HostPtr<int32_t> counts_pin;
    HostPtr<float4> models_pin;
    HostPtr<float> acc_pin;
  } pw;
  // cm_*proceed_zones: stage results parked between the three multi-cloud stages, and the two result clouds
  struct ProceedWs {
    size_t cap = 0;
    DevPtr<float4> low, high, rest, planes;  // [cap] each
    DevPtr<float4> no_ground, ground;        // [2 cap] (windows share their end points)
  } prz;
  // host path: slots and streams are set up together on first use (empty until then)
  std::vector<Slot> slots;
  std::vector<Stream> sensor_stream;
  size_t slot_stride = 0;
  int fill = 0;
  int64_t ticket_counter = 0;
  bool use_graph = true;  // CM_NO_GRAPH=1 switches the frame graphs off
  int submit_policy = CM_SUBMIT_LATEST_WINS;
};

namespace {

int fail(cm_handle_t h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->last_error = buf;
  return code;
}

#define CM_CUDA(h, expr)                                                                              \
  do {                                                                                                \
    cudaError_t e__ = (expr);                                                                         \
    if (e__ != cudaSuccess) return fail(h, CM_E_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                                        __FILE__, __LINE__);                                          \
  } while (0)

// ---- page-locked host memory next to the GPU ---------------------------------------------------------------------------------
// A frame travels host -> device at PCIe speed only if its pages sit on the NUMA node the GPU hangs off: with one process per
// GPU and eight GPUs copying at once, arenas that all landed on one node share that node's memory controllers and the
// inter-socket link. Pages are placed where the allocating thread runs (first touch), so the thread is moved to the CPUs of
// the current device's node for the duration of the allocation (sysfs: /sys/bus/pci/devices/<bdf>/numa_node). A platform
// that does not tell (numa_node = -1, single node, restricted cpuset) gets the plain allocation. CM_NO_NUMA=1 switches it off.
int numa_node_of_current_device() {
  int dev = 0;
  char bus[64] = {0};
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetPCIBusId(bus, (int)sizeof(bus), dev) != cudaSuccess) { cudaGetLastError(); return -1; }
  for (char* c = bus; *c; ++c) *c = (char)tolower(*c);
  char path[160];
  snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
  FILE* f = fopen(path, "r");
  if (!f) return -1;
  int node = -1;
  if (fscanf(f, "%d", &node) != 1) node = -1;
  fclose(f);
  return node;
}
bool cpus_of_node(int node, cpu_set_t* set) {
  char path[96];
  snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
  FILE* f = fopen(path, "r");
  if (!f) return false;
  CPU_ZERO(set);
  int a = 0, b = 0, n = 0;
  char sep = 0;
  while (fscanf(f, "%d", &a) == 1) {
    b = a;
    int c = fgetc(f);
    if (c == '-') { if (fscanf(f, "%d", &b) != 1) break; c = fgetc(f); }
    for (int k = a; k <= b && k < CPU_SETSIZE; ++k) { CPU_SET(k, set); ++n; }
    sep = (char)c;
    if (sep != ',') break;
  }
  fclose(f);
  return n > 0;
}
template <typename T>
cudaError_t pinned_alloc(HostPtr<T>& p, size_t bytes, unsigned flags) {
  static const bool no_numa = getenv("CM_NO_NUMA") != nullptr;
  cpu_set_t old_set, local;
  bool moved = false;
  if (!no_numa) {
    const int node = numa_node_of_current_device();
    if (node >= 0 && cpus_of_node(node, &local) && sched_getaffinity(0, sizeof(old_set), &old_set) == 0) {
      cpu_set_t both;
      CPU_AND(&both, &local, &old_set);  // stay inside what the process is allowed to use
      if (CPU_COUNT(&both) > 0 && !CPU_EQUAL(&both, &old_set)) moved = sched_setaffinity(0, sizeof(both), &both) == 0;
    }
  }
  void* raw = nullptr;
  const cudaError_t e = cudaHostAlloc(&raw, bytes ? bytes : 1, flags);
  if (moved) sched_setaffinity(0, sizeof(old_set), &old_set);
  p.reset(e == cudaSuccess ? static_cast<T*>(raw) : nullptr);
  return e;
}

// `count` elements, at least `min_bytes`
template <typename T>
cudaError_t dev_alloc(DevPtr<T>& p, size_t count, size_t min_bytes = kAlign) {
  void* raw = nullptr;
  const cudaError_t e = cudaMalloc(&raw, std::max<size_t>(count * sizeof(T), min_bytes));
  p.reset(e == cudaSuccess ? static_cast<T*>(raw) : nullptr);
  return e;
}

// An event or stream made by cudaEventCreateWithFlags / cudaStreamCreateWithFlags (left empty if the call fails).
template <typename Owner>
cudaError_t create(Owner& p, cudaError_t (*make)(typename Owner::pointer*, unsigned), unsigned flags) {
  typename Owner::pointer raw = nullptr;
  const cudaError_t e = make(&raw, flags);
  p.reset(e == cudaSuccess ? raw : nullptr);
  return e;
}

int ws_alloc(cm_handle_t h, Workspace& w, uint32_t points, uint32_t frames, uint32_t segs, int out_step) {
  w = Workspace();  // frees what an earlier, failed call left behind
  w.cap_points = points; w.cap_frames = frames; w.cap_segs = segs; w.out_step = out_step;
  w.ml.build(frames, segs);
  const size_t np = std::max<uint32_t>(points, 1);
  CM_CUDA(h, dev_alloc(w.meta, w.ml.total));
  CM_CUDA(h, cudaMemset(w.meta.get(), 0, w.ml.total));
  CM_CUDA(h, pinned_alloc(w.report, w.ml.total, cudaHostAllocDefault));
  memset(w.report.get(), 0, w.ml.total);
  CM_CUDA(h, dev_alloc(w.segs, segs));
  CM_CUDA(h, dev_alloc(w.surv_xyzi, np));
  CM_CUDA(h, dev_alloc(w.surv_src, np));
  CM_CUDA(h, dev_alloc(w.surv_key, np));
  CM_CUDA(h, dev_alloc(w.first_k1, sort_lookback_rows((uint32_t)np)));
  CM_CUDA(h, dev_alloc(w.keys_a, np, 0));
  CM_CUDA(h, dev_alloc(w.keys_b, np, 0));
  CM_CUDA(h, dev_alloc(w.vals_a, np));
  CM_CUDA(h, dev_alloc(w.vals_b, np));
  // every segment owns at least one K1 tile
  w.lb_k1_n = np / k1_min_tile_points() + segs + 2;
  CM_CUDA(h, dev_alloc(w.tile_seg, w.lb_k1_n));
  w.lb_sort_n = (sort_lookback_rows((uint32_t)np) + (frames > 1 ? frames : 0u)) * CM_RADIX;  // segmented: a partial tile per frame
  if (frames > 1) {
    CM_CUDA(h, dev_alloc(w.seg_tile, sort_lookback_rows((uint32_t)np) + frames));
    CM_CUDA(h, dev_alloc(w.seg_hist, (size_t)frames * CM_SEG_PASSES * CM_RADIX));
    CM_CUDA(h, dev_alloc(w.seg_frame_tile0, (size_t)frames + 1));
    CM_CUDA(h, dev_alloc(w.seg_cent_range, np / centroid_tile_items() + 2));
  }
  w.lb_cent_n = np / centroid_tile_items() + 2;
  CM_CUDA(h, dev_alloc(w.tile_rec, w.lb_k1_n));
  CM_CUDA(h, dev_alloc(w.lb_sort, w.lb_sort_n));
  CM_CUDA(h, dev_alloc(w.cent_status, w.lb_cent_n));
  CM_CUDA(h, cudaMemset(w.cent_status.get(), 0, w.lb_cent_n * 8));
  CM_CUDA(h, cudaMemset(w.lb_sort.get(), 0, w.lb_sort_n * 8));
  CM_CUDA(h, dev_alloc(w.epoch_dev, (size_t)1));
  CM_CUDA(h, cudaMemcpy(w.epoch_dev.get(), &h->epoch_start, sizeof(uint32_t), cudaMemcpyHostToDevice));
  CM_CUDA(h, dev_alloc(w.out_xyzi, np * (size_t)out_step, 0));
  CM_CUDA(h, dev_alloc(w.out_count, np));
  CM_CUDA(h, dev_alloc(w.out_idx, np));
  for (auto& e : w.ev) CM_CUDA(h, create(e, cudaEventCreateWithFlags, cudaEventDefault));
  if (getenv("CM_TRACE")) {
    w.trace_k1_n = w.lb_k1_n * 8; w.trace_sort_n = (w.lb_sort_n / CM_RADIX) * 8;
    CM_CUDA(h, dev_alloc(w.trace_k1, w.trace_k1_n));
    CM_CUDA(h, dev_alloc(w.trace_sort, w.trace_sort_n));
    CM_CUDA(h, cudaMemset(w.trace_k1.get(), 0, w.trace_k1_n * 8));
    CM_CUDA(h, cudaMemset(w.trace_sort.get(), 0, w.trace_sort_n * 8));
  }
  // the clears above ran on the default stream: callers may go on with a non-blocking stream of their own
  CM_CUDA(h, cudaDeviceSynchronize());
  w.ready = true;
  return CM_OK;
}

uint32_t seg_mode(const cm_layout_t& L) {
  if (L.point_step == 16 && L.off_x == 0 && L.off_y == 4 && L.off_z == 8 && L.off_intensity == 12) return SEG_PACKED16;
  if (L.point_step == 32 && L.off_x == 0 && L.off_y == 4 && L.off_z == 8 && L.off_intensity == 16) return SEG_PCL32;
  const bool a4 = (L.point_step % 4 == 0) && (L.off_x % 4 == 0) && (L.off_y % 4 == 0) && (L.off_z % 4 == 0) &&
                  (L.off_intensity < 0 || L.off_intensity % 4 == 0);
  if (a4) return SEG_ALIGNED4;
  if (L.point_step <= CM_MAX_STAGED_STEP) return SEG_STAGED;
  return SEG_BYTES;
}

bool layout_ok(const cm_layout_t& L) {
  if (L.point_step < 12 || L.point_step > 65535) return false;
  auto in = [&](int off) { return off >= 0 && off + 4 <= L.point_step; };
  if (!in(L.off_x) || !in(L.off_y) || !in(L.off_z)) return false;
  if (L.off_intensity >= 0 && !in(L.off_intensity)) return false;
  return true;
}

inline uint32_t bits_for(unsigned long long count) {  // bits needed to index `count` distinct values
  uint32_t b = 0;
  while (b < 64 && (count - 1ull) >> b) ++b;
  return count <= 1 ? 0 : b;
}

// Upper bound of the cells of one frame that follows from the crop box alone (no device round trip).
bool crop_cell_bound(cm_handle_t h, unsigned long long* cells) {
  if (h->crop.n_pass <= 0) return false;
  unsigned long long prod = 1;
  for (int a = 0; a < 3; ++a) {
    float lo = -std::numeric_limits<float>::infinity(), hi = std::numeric_limits<float>::infinity();
    for (int k = 0; k < h->crop.n_pass; ++k) {
      const PassDev& ps = h->crop.pass[k];
      if (ps.axis != a || ps.negative) continue;
      if (!(ps.lo == ps.lo) || !(ps.hi == ps.hi)) return false;  // NaN limits bound nothing
      lo = std::max(lo, ps.lo);
      hi = std::min(hi, ps.hi);
    }
    if (!std::isfinite(lo) || !std::isfinite(hi)) return false;
    long long div = 1;
    if (hi >= lo) {
      const float flo = std::floor(lo * h->inv_leaf[a]), fhi = std::floor(hi * h->inv_leaf[a]);
      if (!(std::fabs(flo) < 1e9f) || !(std::fabs(fhi) < 1e9f)) return false;
      div = (long long)fhi - (long long)flo + 1;
    }
    if (div > (1ll << 21)) return false;
    prod *= (unsigned long long)div;
  }
  *cells = prod;
  return true;
}

// The voxel grid of the crop BOX (cm_set_crop chains that are one box bounding x, y and z): it contains the grid PCL derives
// from the data of any frame, so K1 can key the survivors against it (see BoxGrid). false: not a bounding box / too many cells.
bool crop_box_grid(cm_handle_t h, uint32_t n_frames, BoxGrid* g) {
  const CropDev& c = h->crop;
  if (!c.is_box) return false;
  const float fmax = std::numeric_limits<float>::max();
  unsigned long long div[3];
  for (int a = 0; a < 3; ++a) {
    if (!(c.lo[a] > -fmax) || !(c.hi[a] < fmax) || !(c.hi[a] >= c.lo[a])) return false;
    const float flo = std::floor(c.lo[a] * h->inv_leaf[a]), fhi = std::floor(c.hi[a] * h->inv_leaf[a]);
    if (!(std::fabs(flo) < 1e9f) || !(std::fabs(fhi) < 1e9f)) return false;
    g->inv[a] = h->inv_leaf[a];
    g->min_b[a] = (int32_t)flo;
    div[a] = (unsigned long long)((long long)fhi - (long long)flo + 1);
    if (div[a] > (1ull << 21)) return false;
  }
  const unsigned long long cells = div[0] * div[1] * div[2];
  const uint32_t idx_bits = bits_for(cells), bits = idx_bits + bits_for(n_frames);
  if (bits > 32u || cells > 0xFFFFFFFFull) return false;
  g->mul1 = (uint32_t)div[0];
  g->mul2 = (uint32_t)(div[0] * div[1]);
  g->idx_bits = idx_bits;
  g->n_pass = std::max<uint32_t>(1u, (bits + CM_RADIX_BITS - 1) / CM_RADIX_BITS);
  return true;
}

void fill_voxel_params(cm_handle_t h, Workspace& w, VoxelParams& vp, const float4* pts, uint32_t n_frames,
                       uint32_t max_points) {
  vp.pts = pts;
  vp.frame_surv_start = reinterpret_cast<uint32_t*>(w.meta.get() + w.ml.off_fstart);
  vp.n_frames = n_frames;
  vp.max_points = max_points;
  for (int k = 0; k < 3; ++k) vp.inv_leaf[k] = h->inv_leaf[k];
  vp.min_points = h->min_points;
  vp.downsample_all = h->downsample_all;
  vp.pcl_refuses = h->overflow_mode == 1 ? 1u : 0u;
  vp.key_bytes = 8;
  vp.out_step = (uint32_t)w.out_step;
  vp.ctrl = reinterpret_cast<Ctrl*>(w.meta.get() + w.ml.off_ctrl);
  vp.acc = reinterpret_cast<FrameAcc*>(w.meta.get() + w.ml.off_acc);
  vp.grid = reinterpret_cast<GridDev*>(w.meta.get() + w.ml.off_grid);
  vp.info = reinterpret_cast<SortInfo*>(w.meta.get() + w.ml.off_info);
  vp.hist = reinterpret_cast<uint32_t*>(w.meta.get() + w.ml.off_hist);
  vp.keys_a = w.keys_a.get(); vp.keys_b = w.keys_b.get(); vp.vals_a = w.vals_a.get(); vp.vals_b = w.vals_b.get();
  vp.lb_sort = w.lb_sort.get(); vp.cent_status = w.cent_status.get();
  vp.cent_status_words = (uint32_t)std::min<size_t>(w.lb_cent_n, 0xFFFFFFFFu);
  vp.tile_rec = w.ran_k1 ? w.tile_rec.get() : nullptr;
  vp.n_k1_tiles = w.n_k1_tiles;
  vp.epoch_dev = w.epoch_dev.get();
  vp.lb_sort_words = (uint32_t)std::min<size_t>(w.lb_sort_n, 0xFFFFFFFFu);
  vp.max_passes = CM_MAX_SORT_PASSES;
  vp.fused_keys = 0; vp.surv_key = w.surv_key.get(); vp.box = BoxGrid{}; vp.first_k1 = w.first_k1.get();
  vp.sort_tile = sort_tile_items(4, max_points);
  vp.dual_width = 0;
  vp.segmented = 0; vp.seg_tile = w.seg_tile.get(); vp.seg_hist = w.seg_hist.get(); vp.seg_frame_tile0 = w.seg_frame_tile0.get();
  vp.seg_cent_range = w.seg_cent_range.get();
  vp.out_xyzi = w.out_xyzi.get(); vp.out_count = w.out_count.get(); vp.out_idx = w.out_idx.get();
  vp.trace = w.trace_sort.get();
  const char* tp = getenv("CM_TRACE_PASS");
  vp.trace_pass = tp ? (uint32_t)atoi(tp) : 1u;
}

// VoxelGrid stages on vp.pts. bounded: the crop box bounds the key width, so no device round trip is needed.
int run_voxel(cm_handle_t h, Workspace& w, VoxelParams& vp, cudaStream_t st, bool scan_k1_tiles = false,
              bool with_centroid = true, int known_idx_bits = -1) {
  unsigned long long cells = 0;
  // known_idx_bits: the caller already knows an upper bound of the voxel-index width (giant-cloud mode: from the global grid)
  const bool bounded = vp.fused_keys || known_idx_bits >= 0 || (w.ran_k1 && crop_cell_bound(h, &cells));
  if (vp.fused_keys) {  // K1 keyed the survivors against the crop box's grid and counted the digits
    vp.key_bytes = 4;
    vp.max_passes = vp.box.n_pass;
  } else if (bounded) {
    const uint32_t bits = (known_idx_bits >= 0 ? (uint32_t)known_idx_bits : bits_for(cells)) + bits_for(vp.n_frames);
    vp.key_bytes = bits <= 32 ? 4 : 8;
    vp.max_passes = std::max<uint32_t>(1, (bits + CM_RADIX_BITS - 1) / CM_RADIX_BITS);
  } else {
    vp.key_bytes = 8;
    vp.max_passes = CM_MAX_SORT_PASSES;
  }
  // An unbounded grid (no crop box on x, y, z) has its key width decided on the device. For the VoxelGrid proper the host
  // then enqueues BOTH key widths of every kernel and the launches that do not apply exit at once (a dozen empty launches,
  // ~2 us each): no host round trip in the middle of the frame, so cm_merge_frame_async stays asynchronous and the frame
  // can be captured as a CUDA graph like a bounded one. (The radius outlier removal keeps the round trip: it sizes its
  // cell table from the plan.)
  static const bool no_dual = getenv("CM_NO_DUAL") != nullptr;
  const bool dual = !bounded && with_centroid && !no_dual;
  w.dual_width = dual;
  vp.dual_width = dual ? 1u : 0u;
  // Batches of several frames: the frame bits need not be sorted (the input is frame-ordered). Taken where it pays -- fewer
  // passes or 32-bit records instead of 64-bit keys: decided here when the grid is bounded, on the device when it is not
  // (then the 32-bit kernels enqueued are the segmented ones: a batch whose voxel index fits 32 bits never needs frame bits).
  static const bool no_seg = getenv("CM_NO_SEGMENTED") != nullptr;
  vp.segmented = 0;
  if (!no_seg && with_centroid && vp.n_frames > 1 && w.seg_tile && !vp.fused_keys) {
    if (dual) {
      vp.segmented = 1;
    } else if (bounded) {
      const uint32_t ib = known_idx_bits >= 0 ? (uint32_t)known_idx_bits : bits_for(cells), fb = bits_for(vp.n_frames);
      const uint32_t p_seg = std::max<uint32_t>(1, (ib + CM_RADIX_BITS - 1) / CM_RADIX_BITS);
      if (ib <= 32 && (p_seg < vp.max_passes || ib + fb > 32)) {
        vp.segmented = 2;
        vp.key_bytes = 4;
        vp.max_passes = p_seg;
      }
    }
  }
  w.segmented = vp.segmented != 0;
  if (vp.segmented)
    CM_CUDA(h, cudaMemsetAsync(w.seg_hist.get(), 0, (size_t)vp.n_frames * CM_SEG_PASSES * CM_RADIX * sizeof(uint32_t), st));
  if (scan_k1_tiles)
    CM_CUDA(h, launch_grid_setup(vp, st, w.tile_rec.get(), w.n_k1_tiles, w.segs.get(), w.n_segs,
                                 reinterpret_cast<uint32_t*>(w.meta.get() + w.ml.off_segstart)));
  else
    CM_CUDA(h, launch_grid_setup(vp, st));
  ++w.launches;
  if (h->profiling) CM_CUDA(h, cudaEventRecord(w.ev[EV_GRID].get(), st));
  if (dual) {
    w.key_bytes = 0;  // known with the report (fetch_report)
    w.max_passes = CM_MAX_SORT_PASSES;
    VoxelParams v4 = vp, v8 = vp;
    v4.key_bytes = 4; v8.key_bytes = 8;
    CM_CUDA(h, launch_key_hist(v4, st));
    CM_CUDA(h, launch_key_hist(v8, st));
    w.launches += 2;
    if (vp.segmented) {
      CM_CUDA(h, launch_seg_base(v4, st));
      ++w.launches;
    }
    if (h->profiling) CM_CUDA(h, cudaEventRecord(w.ev[EV_KEY].get(), st));
    for (uint32_t ps = 0; ps < 4; ++ps) CM_CUDA(h, launch_sort_pass(v4, (int)ps, st));
    for (uint32_t ps = 0; ps < CM_MAX_SORT_PASSES; ++ps) CM_CUDA(h, launch_sort_pass(v8, (int)ps, st));
    w.launches += 4 + CM_MAX_SORT_PASSES;
    if (h->profiling) CM_CUDA(h, cudaEventRecord(w.ev[EV_SORT].get(), st));
    CM_CUDA(h, launch_centroid(v4, st));
    CM_CUDA(h, launch_centroid(v8, st));
    w.launches += 2 * CM_CENTROID_LAUNCHES;
    if (!w.capturing) CM_CUDA(h, cudaEventRecord(w.ev[EV_CENT].get(), st));
    w.ran_voxel = true;
    return CM_OK;
  }
  if (!bounded) {
    // the key width is only known on the device: fetch the plan (one small round trip), then size the sort to it. The
    // control block comes along in the same copy: its error word says whether every frame's grid was usable.
    SortInfo si;
    Ctrl ctrl;
    CM_CUDA(h, cudaMemcpyAsync(w.report.get(), w.meta.get(), w.ml.off_info + sizeof(SortInfo), cudaMemcpyDeviceToHost, st));
    CM_CUDA(h, cudaStreamSynchronize(st));
    memcpy(&si, w.report.get() + w.ml.off_info, sizeof(si));
    memcpy(&ctrl, w.report.get() + w.ml.off_ctrl, sizeof(ctrl));
    vp.key_bytes = si.total_bits <= 32 ? 4 : 8;
    vp.max_passes = si.num_passes;
    w.plan_idx_bits = si.idx_bits; w.plan_total_bits = si.total_bits; w.plan_error = ctrl.error;
  }
  w.key_bytes = vp.key_bytes;
  w.max_passes = vp.max_passes;
  if (!vp.fused_keys) {
    CM_CUDA(h, launch_key_hist(vp, st));
    ++w.launches;
  }
  if (vp.segmented) {
    CM_CUDA(h, launch_seg_base(vp, st));
    ++w.launches;
  }
  if (h->profiling) CM_CUDA(h, cudaEventRecord(w.ev[EV_KEY].get(), st));
  w.timed_pass0 = false;
  for (uint32_t ps = 0; ps < vp.max_passes; ++ps) {
    CM_CUDA(h, launch_sort_pass(vp, (int)ps, st));
    ++w.launches;
    if (ps == 0 && h->profiling) {  // pass 0 of a fused-key run does the key kernel's histogram work too: timed on its own
      CM_CUDA(h, cudaEventRecord(w.ev[EV_SORT0].get(), st));
      w.timed_pass0 = true;
    }
  }
  if (h->profiling) CM_CUDA(h, cudaEventRecord(w.ev[EV_SORT].get(), st));
  if (!with_centroid) {  // the caller only wants the points sorted by cell (radius outlier removal)
    w.ran_voxel = false;
    return CM_OK;
  }
  CM_CUDA(h, launch_centroid(vp, st));
  w.launches += CM_CENTROID_LAUNCHES;
  if (!w.capturing) CM_CUDA(h, cudaEventRecord(w.ev[EV_CENT].get(), st));
  w.ran_voxel = true;
  return CM_OK;
}

// Derives the single-box form of a PassThrough chain (CropDev, ZoneDev) whenever the chain allows it.
template <typename Chain>
void derive_box(Chain& c) {
  const float fmax = std::numeric_limits<float>::max();
  c.is_box = 0; c.use_i = 0;
  for (int a = 0; a < 4; ++a) { c.lo[a] = -fmax; c.hi[a] = fmax; }
  if (c.n_pass <= 0) return;
  for (int k = 0; k < c.n_pass; ++k) {
    const PassDev& ps = c.pass[k];
    if (ps.negative || !(ps.lo == ps.lo) || !(ps.hi == ps.hi)) return;  // negative window or NaN limit: general chain
    c.lo[ps.axis] = std::max(c.lo[ps.axis], ps.lo);
    c.hi[ps.axis] = std::min(c.hi[ps.axis], ps.hi);
    if (ps.axis == 3) c.use_i = 1;
  }
  c.is_box = 1;
}

struct SegPlan {
  uint32_t n_frames = 0, n_tiles = 0, tile_points = 0, tiles_per_seg = 0, staged_smem = 0;
  int mode = -1;
  int64_t total_points = 0;
};

// Build the device segment table for a batch.
int build_segments(cm_handle_t h, Workspace& w, const cm_segment_t* segs, int n_seg, std::vector<SegDev>& out,
                   std::vector<uint32_t>& tile_seg, SegPlan* plan) {
  if (n_seg <= 0 || !segs) return fail(h, CM_E_INVALID, "no segments");
  if ((uint32_t)n_seg > w.cap_segs) return fail(h, CM_E_CAPACITY, "%d segments > capacity %u", n_seg, w.cap_segs);
  int64_t total = 0;
  uint32_t max_step_staged = 0;
  int common_mode = -2;
  for (int s = 0; s < n_seg; ++s) {
    const cm_segment_t& g = segs[s];
    if (!layout_ok(g.layout)) return fail(h, CM_E_INVALID, "segment %d: bad layout", s);
    if (g.n_points < 0 || g.n_points > 0xFFFFFFF0ll) return fail(h, CM_E_INVALID, "segment %d: bad n_points", s);
    if (g.n_points > 0 && (!g.data || (reinterpret_cast<uintptr_t>(g.data) & 15u)))
      return fail(h, CM_E_INVALID, "segment %d: data must be a 16-byte aligned device pointer", s);
    if (g.sensor < 0 || g.sensor >= h->cfg.max_sensors) return fail(h, CM_E_INVALID, "segment %d: bad sensor", s);
    if (s == 0 ? g.frame != 0 : (g.frame != segs[s - 1].frame && g.frame != segs[s - 1].frame + 1))
      return fail(h, CM_E_INVALID, "segment %d: frames must start at 0 and increase by steps of 1", s);
    const int md = (int)seg_mode(g.layout);
    if (md == (int)SEG_STAGED) max_step_staged = std::max<uint32_t>(max_step_staged, (uint32_t)g.layout.point_step);
    common_mode = (common_mode == -2 || common_mode == md) ? md : -1;
    total += g.n_points;
  }
  if (total > (int64_t)w.cap_points) return fail(h, CM_E_CAPACITY, "%lld points > capacity %u", (long long)total, w.cap_points);
  uint32_t T = k1_tile_points(total);
  if (max_step_staged && k1_staged_smem(T, max_step_staged) > 200u * 1024u) T = k1_min_tile_points();
  out.resize(n_seg);
  uint32_t tile = 0, frame = 0, src_base = 0;
  uint64_t slot_base = 0;
  bool uniform = true;
  uint32_t tps = 0;
  for (int s = 0; s < n_seg; ++s) {
    const cm_segment_t& g = segs[s];
    const bool first = (s == 0) || (g.frame != segs[s - 1].frame);
    if (first) { frame = (uint32_t)g.frame; src_base = 0; }
    SegDev& d = out[s];
    memset(&d, 0, sizeof(d));
    d.data = static_cast<const uint8_t*>(g.data);
    d.n_points = (uint32_t)g.n_points;
    d.tile_begin = tile;
    d.src_base = src_base;
    d.slot_base = (uint32_t)slot_base;
    d.frame = frame;
    d.point_step = g.layout.point_step;
    d.off_x = g.layout.off_x; d.off_y = g.layout.off_y; d.off_z = g.layout.off_z;
    d.off_i = g.layout.off_intensity >= 0 ? g.layout.off_intensity : -1;
    d.is_dense = g.layout.is_dense ? 1u : 0u;
    d.sensor = (uint32_t)g.sensor;
    d.first_of_frame = first ? 1u : 0u;
    d.mode = seg_mode(g.layout);
    memcpy(d.m, h->mats_host + g.sensor * 12, sizeof(d.m));
    const uint32_t nt = std::max<uint32_t>(1u, (d.n_points + T - 1) / T);
    if (s == 0) tps = nt; else if (nt != tps) uniform = false;
    tile += nt;
    src_base += d.n_points;
    slot_base += d.n_points;
  }
  if (frame + 1 > w.cap_frames) return fail(h, CM_E_CAPACITY, "%u frames > capacity %u", frame + 1, w.cap_frames);
  if ((size_t)tile + 1 > w.lb_k1_n) return fail(h, CM_E_CAPACITY, "too many tiles");
  if (slot_base > 0xFFFFFFF0ull) return fail(h, CM_E_CAPACITY, "batch too large");
  tile_seg.clear();
  if (!uniform) {
    tile_seg.resize(tile);
    for (int s = 0; s < n_seg; ++s) {
      const uint32_t te = (s + 1 < n_seg) ? out[s + 1].tile_begin : tile;
      for (uint32_t t = out[s].tile_begin; t < te; ++t) tile_seg[t] = (uint32_t)s;
    }
  }
  plan->n_frames = frame + 1; plan->n_tiles = tile; plan->tile_points = T; plan->total_points = total;
  plan->tiles_per_seg = uniform ? tps : 0u;
  plan->mode = (common_mode == (int)SEG_PACKED16 || common_mode == (int)SEG_PCL32) ? common_mode : -1;
  plan->staged_smem = max_step_staged ? k1_staged_smem(T, max_step_staged) : 0u;
  return CM_OK;
}

int run_pipeline(cm_handle_t h, Workspace& w, const cm_segment_t* segs, int n_seg, cudaStream_t st, bool with_voxel) {
  SegPlan plan;
  std::vector<SegDev> sd;
  std::vector<uint32_t> ts;
  int rc = build_segments(h, w, segs, n_seg, sd, ts, &plan);
  if (rc != CM_OK) return rc;
  if (sd.size() != w.segs_host.size() || memcmp(sd.data(), w.segs_host.data(), sd.size() * sizeof(SegDev)) != 0) {
    CM_CUDA(h, cudaMemcpyAsync(w.segs.get(), sd.data(), sd.size() * sizeof(SegDev), cudaMemcpyHostToDevice, st));
    w.segs_host = sd;
  }
  if (!ts.empty() && ts != w.tile_seg_host) {
    CM_CUDA(h, cudaMemcpyAsync(w.tile_seg.get(), ts.data(), ts.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    w.tile_seg_host = ts;
  }
  const uint32_t n_frames = plan.n_frames;
  const int64_t total = plan.total_points;
  w.has_run = true; w.report_valid = false; w.profiled = h->profiling;
  w.n_frames = n_frames; w.n_segs = (uint32_t)n_seg; w.points_in = total; w.launches = 0;
  w.ran_k1 = true; w.ran_voxel = false; w.stream = st;
  w.voxel_pts = w.surv_xyzi.get();
  h->last = &w;

  if (!w.capturing) CM_CUDA(h, cudaEventRecord(w.ev[EV_START].get(), st));
  CM_CUDA(h, cudaMemsetAsync(w.meta.get(), 0, w.ml.zero_bytes, st));
  K1Params kp;
  kp.segs = w.segs.get(); kp.n_seg = (uint32_t)n_seg; kp.n_tiles = plan.n_tiles; kp.n_frames = n_frames;
  kp.tiles_per_seg = plan.tiles_per_seg; kp.tile_seg = w.tile_seg.get();
  kp.crop = h->crop;
  kp.surv_xyzi = w.surv_xyzi.get(); kp.surv_src = w.surv_src.get();
  kp.ctrl = reinterpret_cast<Ctrl*>(w.meta.get() + w.ml.off_ctrl);
  kp.acc = reinterpret_cast<FrameAcc*>(w.meta.get() + w.ml.off_acc);
  kp.tile_rec = w.tile_rec.get();
  kp.trace = w.trace_k1.get();
  // K1 keys the survivors itself when the crop is a box that bounds the grid (no k_voxel_key_hist): CM_NO_FUSED_KEYS=1 keeps
  // the separate key kernel (A/B and test hook)
  static const bool no_fused = getenv("CM_NO_FUSED_KEYS") != nullptr;
  BoxGrid box{};
  const bool fused = with_voxel && !no_fused && crop_box_grid(h, n_frames, &box);
  w.fused_keys = fused; w.box = box;
  kp.surv_key = fused ? w.surv_key.get() : nullptr;
  kp.hist = reinterpret_cast<uint32_t*>(w.meta.get() + w.ml.off_hist);
  kp.box = box;
  kp.obox = nullptr; kp.n_obox = 0;
  if (h->n_obox > 0) {  // the stage table travels like the segment table: uploaded on the run's stream when it changed
    const std::vector<OrientedBoxDev> ob(h->obox, h->obox + h->n_obox);
    if (!w.obox) CM_CUDA(h, dev_alloc(w.obox, CM_MAX_CROP_BOXES));
    if (ob.size() != w.obox_host.size() || memcmp(ob.data(), w.obox_host.data(), ob.size() * sizeof(OrientedBoxDev)) != 0) {
      CM_CUDA(h, cudaMemcpyAsync(w.obox.get(), ob.data(), ob.size() * sizeof(OrientedBoxDev), cudaMemcpyHostToDevice, st));
      w.obox_host = ob;
    }
    kp.obox = w.obox.get(); kp.n_obox = (uint32_t)h->n_obox;
  }
  w.n_k1_tiles = plan.n_tiles;
  w.dense_valid = false;
  CM_CUDA(h, launch_transform_crop(kp, plan.tile_points, plan.mode, plan.staged_smem, st));
  ++w.launches;
  if (!with_voxel) {
    CM_CUDA(h, launch_tile_scan(w.tile_rec.get(), plan.n_tiles, w.segs.get(), (uint32_t)n_seg, n_frames,
                                reinterpret_cast<uint32_t*>(w.meta.get() + w.ml.off_fstart),
                                reinterpret_cast<uint32_t*>(w.meta.get() + w.ml.off_segstart), st));
    ++w.launches;
    CM_CUDA(h, cudaEventRecord(w.ev[EV_K1].get(), st));
    return CM_OK;
  }
  if (!w.capturing) CM_CUDA(h, cudaEventRecord(w.ev[EV_K1].get(), st));
  VoxelParams vp;
  fill_voxel_params(h, w, vp, w.surv_xyzi.get(), n_frames, (uint32_t)total);
  vp.fused_keys = fused ? 1u : 0u;
  vp.box = box;
  return run_voxel(h, w, vp, st, true);  // the tile scan rides in the grid-setup launch
}

// Dense copy of the merged cropped cloud of the last K1 run (allocated on first use).
int materialize_dense(cm_handle_t h, Workspace& w) {
  if (!w.ran_k1 || w.dense_valid) return CM_OK;
  const size_t np = std::max<uint32_t>(w.cap_points, 1);
  if (!w.dense_xyzi) {  // all three or none
    DevPtr<float4> xyzi; DevPtr<uint32_t> src, slot;
    CM_CUDA(h, dev_alloc(xyzi, np));
    CM_CUDA(h, dev_alloc(src, np));
    CM_CUDA(h, dev_alloc(slot, np));
    w.dense_xyzi = std::move(xyzi); w.dense_src = std::move(src); w.dense_slot = std::move(slot);
  }
  CM_CUDA(h, launch_compact_survivors(w.tile_rec.get(), w.n_k1_tiles, w.surv_xyzi.get(), w.surv_src.get(), w.dense_xyzi.get(),
                                      w.dense_src.get(), w.dense_slot.get(), w.stream));
  w.dense_valid = true;
  return CM_OK;
}

// D2H of the control block of the last run + decode into stats / frame info. Blocks.
int fetch_report(cm_handle_t h, Workspace& w, cudaEvent_t already_copied = nullptr) {
  if (!w.has_run) return fail(h, CM_E_INVALID, "nothing has run on this handle");
  if (w.report_valid) return CM_OK;
  if (already_copied) {
    CM_CUDA(h, cudaEventSynchronize(already_copied));  // the run enqueued the report copy itself
  } else {
    CM_CUDA(h, cudaMemcpyAsync(w.report.get(), w.meta.get(), w.ml.total, cudaMemcpyDeviceToHost, w.stream));
    CM_CUDA(h, cudaStreamSynchronize(w.stream));
  }
  const Ctrl* ctrl = reinterpret_cast<const Ctrl*>(w.report.get() + w.ml.off_ctrl);
  const FrameAcc* acc = reinterpret_cast<const FrameAcc*>(w.report.get() + w.ml.off_acc);
  const SortInfo* si = reinterpret_cast<const SortInfo*>(w.report.get() + w.ml.off_info);
  const uint32_t* fstart = reinterpret_cast<const uint32_t*>(w.report.get() + w.ml.off_fstart);
  const GridDev* grid = reinterpret_cast<const GridDev*>(w.report.get() + w.ml.off_grid);
  cm_stats_t& s = h->stats;
  memset(&s, 0, sizeof(s));
  s.points_in = w.points_in;
  s.frames = (int32_t)w.n_frames;
  s.survivors = fstart[w.n_frames];
  s.device_error = (int32_t)ctrl->error;
  h->frame_info.assign(w.n_frames, cm_frame_info_t{});
  int64_t vbeg = 0;
  for (uint32_t f = 0; f < w.n_frames; ++f) {
    cm_frame_info_t& fi = h->frame_info[f];
    fi.survivor_begin = fstart[f];
    fi.survivor_end = fstart[f + 1];
    if (w.ran_voxel) {
      fi.voxel_begin = vbeg;
      vbeg += acc[f].voxel_count;
      fi.voxel_end = vbeg;
      for (int k = 0; k < 3; ++k) { fi.min_b[k] = grid[f].min_b[k]; fi.max_b[k] = grid[f].max_b[k]; fi.div_b[k] = grid[f].div_b[k]; }
      fi.pcl_overflow = grid[f].pcl_overflow;
      s.pcl_overflow += grid[f].pcl_overflow;
    }
  }
  if (w.ran_voxel) {
    s.voxels_out = ctrl->total_voxels;
    s.key_bits = (int32_t)si->total_bits;
    s.sort_passes = (int32_t)si->num_passes;
    if (w.dual_width) w.key_bytes = si->width == 4u ? 4u : 8u;
    s.key_bytes = (int32_t)w.key_bytes;
  }
  const int last_ev = w.ran_voxel ? EV_CENT : EV_K1;
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, w.ev[EV_START].get(), w.ev[last_ev].get()) == cudaSuccess) s.gpu_ms = ms;
  else cudaGetLastError();  // a failed query must not surface later as the result of an unrelated launch
  for (auto& v : h->stage_ms) v = -1.f;
  h->stage_ms[EV_START] = s.gpu_ms;
  if (w.profiled) {
    float t;
    if (cudaEventElapsedTime(&t, w.ev[EV_START].get(), w.ev[EV_K1].get()) == cudaSuccess) h->stage_ms[EV_K1] = t;
    if (w.ran_voxel) {
      if (cudaEventElapsedTime(&t, w.ev[EV_K1].get(), w.ev[EV_GRID].get()) == cudaSuccess) h->stage_ms[EV_GRID] = t;
      if (cudaEventElapsedTime(&t, w.ev[EV_GRID].get(), w.ev[EV_KEY].get()) == cudaSuccess) h->stage_ms[EV_KEY] = t;
      if (cudaEventElapsedTime(&t, w.ev[EV_KEY].get(), w.ev[EV_SORT].get()) == cudaSuccess) h->stage_ms[EV_SORT] = t;
      if (w.timed_pass0 && cudaEventElapsedTime(&t, w.ev[EV_KEY].get(), w.ev[EV_SORT0].get()) == cudaSuccess) h->stage_ms[EV_SORT0] = t;
      if (cudaEventElapsedTime(&t, w.ev[EV_SORT].get(), w.ev[EV_CENT].get()) == cudaSuccess) h->stage_ms[EV_CENT] = t;
    }
  }
  w.report_valid = true;
  if (ctrl->error == CM_DEV_E_KEY_RANGE) return fail(h, CM_E_KEY_RANGE, "voxel grid exceeds the key range (leaf too small for the extent)");
  if (ctrl->error) return fail(h, CM_E_INTERNAL, "device watchdog tripped (code %u)", ctrl->error);
  return CM_OK;
}

int ensure_batch_ws(cm_handle_t h) {
  if (h->batch.ready) return CM_OK;
  const cm_config_t& c = h->cfg;
  return ws_alloc(h, h->batch, (uint32_t)c.max_batch_points, (uint32_t)c.max_batch_frames, (uint32_t)c.max_batch_segments,
                  c.out_point_step);
}

// Sets up the slots and the sensor streams in locals and commits them only when all of it succeeded: a failure leaves the
// handle as it was, and the slots never move once a run (h->last, a captured graph) can point into them.
int ensure_host_path(cm_handle_t h) {
  if (!h->slots.empty()) return CM_OK;
  const cm_config_t& c = h->cfg;
  h->slot_stride = align_up((size_t)c.max_points_per_sensor * (size_t)c.max_point_step + 16, kAlign);
  std::vector<Stream> streams(c.max_sensors);
  for (auto& s : streams) CM_CUDA(h, create(s, cudaStreamCreateWithFlags, cudaStreamNonBlocking));
  std::vector<Slot> slots(c.frames_in_flight);
  const uint64_t pts = (uint64_t)c.max_sensors * (uint64_t)c.max_points_per_sensor;
  if (pts > 0xFFFFFFF0ull) return fail(h, CM_E_CAPACITY, "max_sensors * max_points_per_sensor too large");
  for (auto& sl : slots) {
    int rc = ws_alloc(h, sl.ws, (uint32_t)pts, 1, (uint32_t)c.max_sensors, c.out_point_step);
    if (rc != CM_OK) return rc;
    CM_CUDA(h, dev_alloc(sl.raw_dev, h->slot_stride * c.max_sensors, 0));
    CM_CUDA(h, pinned_alloc(sl.raw_pinned, h->slot_stride * c.max_sensors, cudaHostAllocDefault));
    sl.arena_bytes = 2 * h->slot_stride * c.max_sensors;
    CM_CUDA(h, dev_alloc(sl.arena_dev, sl.arena_bytes, 0));
    sl.exp_cap = (uint32_t)pts;
    const size_t ecap = std::max<size_t>(sl.exp_cap, 1);
    CM_CUDA(h, pinned_alloc(sl.exp_xyzi, ecap * (size_t)c.out_point_step, cudaHostAllocMapped));
    CM_CUDA(h, pinned_alloc(sl.exp_count, ecap * sizeof(uint32_t), cudaHostAllocMapped));
    CM_CUDA(h, pinned_alloc(sl.exp_idx, ecap * sizeof(unsigned long long), cudaHostAllocMapped));
    sl.sensor.resize(c.max_sensors);
    for (auto& ss : sl.sensor) CM_CUDA(h, create(ss.copied, cudaEventCreateWithFlags, cudaEventDisableTiming));
    CM_CUDA(h, create(sl.stream, cudaStreamCreateWithFlags, cudaStreamNonBlocking));
    CM_CUDA(h, create(sl.done, cudaEventCreateWithFlags, cudaEventDisableTiming));
  }
  h->sensor_stream = std::move(streams);
  h->slots = std::move(slots);
  return CM_OK;
}

int submit_impl(cm_handle_t h, int sensor, const void* data, int64_t n_points, const cm_layout_t* layout, uint64_t stamp,
                bool pinned_src) {
  if (!h) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  if (sensor < 0 || sensor >= h->cfg.max_sensors) return fail(h, CM_E_INVALID, "sensor %d out of range", sensor);
  if (!layout || !layout_ok(*layout)) return fail(h, CM_E_INVALID, "bad layout");
  if (n_points < 0 || (n_points > 0 && !data)) return fail(h, CM_E_INVALID, "bad cloud");
  if (n_points > h->cfg.max_points_per_sensor) return fail(h, CM_E_CAPACITY, "cloud of %lld points > max_points_per_sensor", (long long)n_points);
  if (layout->point_step > h->cfg.max_point_step) return fail(h, CM_E_CAPACITY, "point_step %d > max_point_step", layout->point_step);
  int rc = ensure_host_path(h);
  if (rc != CM_OK) return rc;
  Slot& sl = h->slots[h->fill];
  if (sl.busy) return fail(h, CM_E_CAPACITY, "all %d frame slots are in flight: call cm_wait_frame first", h->cfg.frames_in_flight);
  SensorState& ss = sl.sensor[sensor];
  // the reference's flag gate `if (!flag_x) { store; flag_x = true; }` (pc_preprocessing_main.cpp:330): a cloud that
  // arrives while the sensor's previous one is still waiting to be fused is dropped
  if (h->submit_policy == CM_SUBMIT_FIRST_WINS && ss.submitted) return CM_OK;
  const size_t bytes = (size_t)n_points * (size_t)layout->point_step;
  uint8_t* dst = sl.raw_dev.get() + (size_t)sensor * h->slot_stride;
  cudaStream_t st = h->sensor_stream[sensor].get();
  if (bytes) {
    if (pinned_src) {
      CM_CUDA(h, cudaMemcpyAsync(dst, data, bytes, cudaMemcpyHostToDevice, st));
    } else {
      uint8_t* stg = sl.raw_pinned.get() + (size_t)sensor * h->slot_stride;
      CM_CUDA(h, cudaEventSynchronize(ss.copied.get()));  // the previous copy out of this staging buffer is done
      memcpy(stg, data, bytes);
      CM_CUDA(h, cudaMemcpyAsync(dst, stg, bytes, cudaMemcpyHostToDevice, st));
    }
  }
  CM_CUDA(h, cudaEventRecord(ss.copied.get(), st));
  ss.submitted = true; ss.n_points = n_points; ss.layout = *layout; ss.stamp = stamp; ss.dev = dst;
  return CM_OK;
}

// Tail of a host-path frame on its stream: the voxels go to the slot's page-locked mirrors (k_export_voxels, sized by the
// device-resident voxel count) and the control block to the pinned report -- both before the frame's `done` event, so
// cm_wait_frame synchronises once and copies nothing over PCIe itself.
cudaError_t enqueue_frame_export(cm_handle_t h, Slot& sl) {
  Workspace& w = sl.ws;
  VoxelParams vp;
  fill_voxel_params(h, w, vp, w.surv_xyzi.get(), 1, 0);
  void *dx = nullptr, *dc = nullptr, *di = nullptr;
  cudaError_t e = cudaHostGetDevicePointer(&dx, sl.exp_xyzi.get(), 0);
  if (e == cudaSuccess) e = cudaHostGetDevicePointer(&dc, sl.exp_count.get(), 0);
  if (e == cudaSuccess) e = cudaHostGetDevicePointer(&di, sl.exp_idx.get(), 0);
  if (e == cudaSuccess) e = launch_export_voxels(vp, dx, static_cast<uint32_t*>(dc), static_cast<unsigned long long*>(di), sl.exp_cap, sl.stream.get());
  if (e != cudaSuccess) return e;
  ++w.launches;
  return cudaMemcpyAsync(w.report.get(), w.meta.get(), w.ml.total, cudaMemcpyDeviceToHost, sl.stream.get());
}

int merge_async_impl(cm_handle_t h, uint64_t mask, int64_t* ticket) {
  int rc = ensure_host_path(h);
  if (rc != CM_OK) return rc;
  Slot& sl = h->slots[h->fill];
  if (sl.busy) return fail(h, CM_E_CAPACITY, "frame slot still in flight");
  cudaStream_t st = sl.stream.get();
  std::vector<cm_segment_t> segs;
  uint64_t used = 0, stamp = 0;
  for (int s = 0; s < h->cfg.max_sensors; ++s) {
    if (!((mask >> s) & 1ull)) continue;
    SensorState& ss = sl.sensor[s];
    if (!ss.submitted) continue;
    cm_segment_t g;
    g.data = ss.dev;
    g.n_points = ss.n_points; g.layout = ss.layout; g.sensor = s; g.frame = 0;
    segs.push_back(g);
    used |= 1ull << s;
    stamp = std::max(stamp, ss.stamp);  // operator+= keeps the newest stamp
    CM_CUDA(h, cudaStreamWaitEvent(st, ss.copied.get(), 0));
  }
  if (segs.empty()) return fail(h, CM_E_NOT_READY, "no submitted cloud for any sensor in the mask");
  // ---- replay / capture / plain enqueue ---------------------------------------------------------------------------------
  // (an unbounded grid is as capturable as a bounded one: its key width is resolved on the device, see run_voxel)
  bool graphable = h->use_graph && !h->profiling;
  std::string key;
  if (graphable) {
    key.assign(reinterpret_cast<const char*>(segs.data()), segs.size() * sizeof(cm_segment_t));
    for (const cm_segment_t& g : segs) key.append(reinterpret_cast<const char*>(h->mats_host + g.sensor * 12), 12 * sizeof(float));
    key.append(reinterpret_cast<const char*>(&h->crop), sizeof(h->crop));
    key.append(reinterpret_cast<const char*>(&h->n_obox), sizeof(h->n_obox));  // the graph reads the stage table uploaded
    key.append(reinterpret_cast<const char*>(h->obox), h->n_obox * sizeof(OrientedBoxDev));  // by the run it was captured in
    key.append(reinterpret_cast<const char*>(h->inv_leaf), sizeof(h->inv_leaf));
    key.append(reinterpret_cast<const char*>(&h->min_points), sizeof(h->min_points));
    key.append(reinterpret_cast<const char*>(&h->downsample_all), sizeof(h->downsample_all));
    key.append(reinterpret_cast<const char*>(&h->overflow_mode), sizeof(h->overflow_mode));  // read by k_grid_setup
  }
  bool launched = false;
  if (graphable && sl.graph && sl.graph_key == key) {
    Workspace& w = sl.ws;  // same configuration as the captured frame: every host-side field of the run is unchanged
    w.has_run = true; w.report_valid = false; w.dense_valid = false; w.stream = st;
    h->last = &w;
    CM_CUDA(h, cudaEventRecord(w.ev[EV_START].get(), st));
    CM_CUDA(h, cudaGraphLaunch(sl.graph.get(), st));
    CM_CUDA(h, cudaEventRecord(w.ev[EV_CENT].get(), st));
    launched = true;
  } else if (graphable && sl.graph_seen == key) {
    // second frame with this configuration (its segment table is already on the device): capture, instantiate, launch
    sl.graph.reset(); sl.graph_key.clear();
    cudaGraph_t g = nullptr;
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed) == cudaSuccess) {
      sl.ws.capturing = true;
      rc = run_pipeline(h, sl.ws, segs.data(), (int)segs.size(), st, true);
      sl.ws.capturing = false;
      cudaError_t ce = cudaSuccess;
      if (rc == CM_OK) ce = enqueue_frame_export(h, sl);
      const cudaError_t ee = cudaStreamEndCapture(st, &g);
      cudaGraphExec_t exec = nullptr;
      if (rc == CM_OK && ce == cudaSuccess && ee == cudaSuccess && g &&
          cudaGraphInstantiate(&exec, g, 0) == cudaSuccess) {
        sl.graph.reset(exec);
        sl.graph_key = key;
        cudaGraphDestroy(g);
        CM_CUDA(h, cudaEventRecord(sl.ws.ev[EV_START].get(), st));
        CM_CUDA(h, cudaGraphLaunch(sl.graph.get(), st));
        CM_CUDA(h, cudaEventRecord(sl.ws.ev[EV_CENT].get(), st));
        launched = true;
      } else {
        if (g) cudaGraphDestroy(g);
        h->use_graph = false;  // not capturable here: stay on the plain path
        cudaGetLastError();
      }
    } else {
      h->use_graph = false;
      cudaGetLastError();
    }
  }
  if (!launched) {
    if (sl.graph && sl.graph_key != key) { sl.graph.reset(); sl.graph_key.clear(); }
    rc = run_pipeline(h, sl.ws, segs.data(), (int)segs.size(), st, true);
    if (rc != CM_OK) return rc;
    CM_CUDA(h, enqueue_frame_export(h, sl));
    sl.graph_seen = key;
  }
  CM_CUDA(h, cudaEventRecord(sl.done.get(), st));
  // Every submission of this slot ends here: merged clouds are consumed; a cloud submitted for a sensor outside the mask is
  // discarded (it would otherwise resurface, stale, when the slot comes round again frames_in_flight frames later).
  for (int s = 0; s < h->cfg.max_sensors; ++s) sl.sensor[s].submitted = false;
  sl.arena_used = 0;
  sl.busy = true; sl.used_mask = used; sl.stamp = stamp;
  sl.ticket = ++h->ticket_counter;
  *ticket = sl.ticket;
  h->fill = (h->fill + 1) % (int)h->slots.size();
  return CM_OK;
}

int wait_impl(cm_handle_t h, int64_t ticket, cm_frame_out_t* out, uint64_t* used_mask, uint64_t* out_stamp) {
  Slot* sl = nullptr;
  for (auto& s : h->slots) if (s.busy && s.ticket == ticket) sl = &s;
  if (!sl) return fail(h, CM_E_INVALID, "unknown ticket %lld", (long long)ticket);
  Workspace& w = sl->ws;
  h->last = &w;
  int rc = fetch_report(h, w, sl->done.get());
  sl->busy = false;
  if (rc != CM_OK) return rc;
  if (used_mask) *used_mask = sl->used_mask;
  if (out_stamp) *out_stamp = sl->stamp;
  if (!out) return CM_OK;
  const cm_frame_info_t& fi = h->frame_info[0];
  out->info = fi;
  out->n_survivors = fi.survivor_end - fi.survivor_begin;
  out->n_voxels = fi.voxel_end - fi.voxel_begin;
  const bool pcl_refuses = h->overflow_mode == 1 && fi.pcl_overflow;
  if (pcl_refuses) out->n_voxels = out->n_survivors;  // PCL 1.8.1: output = *input_
  if ((out->voxel_xyzi || out->voxel_count || out->voxel_idx) && out->n_voxels > out->voxel_capacity)
    return fail(h, CM_E_CAPACITY, "voxel_capacity %lld < %lld voxels", (long long)out->voxel_capacity, (long long)out->n_voxels);
  if ((out->survivor_xyzi || out->survivor_src) && out->n_survivors > out->survivor_capacity)
    return fail(h, CM_E_CAPACITY, "survivor_capacity %lld < %lld survivors", (long long)out->survivor_capacity, (long long)out->n_survivors);
  cudaStream_t st = sl->stream.get();
  const size_t nv = (size_t)out->n_voxels, ns = (size_t)out->n_survivors;
  if ((out->survivor_xyzi || out->survivor_src || pcl_refuses) && ns) {
    rc = materialize_dense(h, w);
    if (rc != CM_OK) return rc;
  }
  if (pcl_refuses) {
    if (out->voxel_xyzi && nv) {
      if (w.out_step == 16) {
        CM_CUDA(h, cudaMemcpyAsync(out->voxel_xyzi, w.dense_xyzi.get(), nv * 16, cudaMemcpyDeviceToHost, st));
      } else {
        // expand packed survivors into pcl::PointXYZI records on the host side of the copy
        std::vector<float> tmp(nv * 4);
        CM_CUDA(h, cudaMemcpyAsync(tmp.data(), w.dense_xyzi.get(), nv * 16, cudaMemcpyDeviceToHost, st));
        CM_CUDA(h, cudaStreamSynchronize(st));
        float* o = static_cast<float*>(out->voxel_xyzi);
        for (size_t i = 0; i < nv; ++i) {
          o[i * 8 + 0] = tmp[i * 4 + 0]; o[i * 8 + 1] = tmp[i * 4 + 1]; o[i * 8 + 2] = tmp[i * 4 + 2]; o[i * 8 + 3] = 1.0f;
          o[i * 8 + 4] = tmp[i * 4 + 3]; o[i * 8 + 5] = 0.f; o[i * 8 + 6] = 0.f; o[i * 8 + 7] = 0.f;
        }
      }
    }
    if (out->voxel_count) for (size_t i = 0; i < nv; ++i) out->voxel_count[i] = 1;
    if (out->voxel_idx) for (size_t i = 0; i < nv; ++i) out->voxel_idx[i] = 0;
  } else if (nv <= (size_t)sl->exp_cap) {
    // the frame's own stream already wrote the voxels to the slot's page-locked mirrors (k_export_voxels): plain memcpy
    if (out->voxel_xyzi && nv) memcpy(out->voxel_xyzi, sl->exp_xyzi.get(), nv * (size_t)w.out_step);
    if (out->voxel_count && nv) memcpy(out->voxel_count, sl->exp_count.get(), nv * 4);
    if (out->voxel_idx && nv) memcpy(out->voxel_idx, sl->exp_idx.get(), nv * 8);
    if (!((out->survivor_xyzi || out->survivor_src) && ns)) return CM_OK;
  } else {
    if (out->voxel_xyzi && nv) CM_CUDA(h, cudaMemcpyAsync(out->voxel_xyzi, w.out_xyzi.get(), nv * (size_t)w.out_step, cudaMemcpyDeviceToHost, st));
    if (out->voxel_count && nv) CM_CUDA(h, cudaMemcpyAsync(out->voxel_count, w.out_count.get(), nv * 4, cudaMemcpyDeviceToHost, st));
    if (out->voxel_idx && nv) CM_CUDA(h, cudaMemcpyAsync(out->voxel_idx, w.out_idx.get(), nv * 8, cudaMemcpyDeviceToHost, st));
  }
  if (out->survivor_xyzi && ns) CM_CUDA(h, cudaMemcpyAsync(out->survivor_xyzi, w.dense_xyzi.get(), ns * 16, cudaMemcpyDeviceToHost, st));
  if (out->survivor_src && ns) CM_CUDA(h, cudaMemcpyAsync(out->survivor_src, w.dense_src.get(), ns * 4, cudaMemcpyDeviceToHost, st));
  CM_CUDA(h, cudaStreamSynchronize(st));
  return CM_OK;
}

}  // namespace

extern "C" {

const char* cm_version(void) { return "cloud_merger_b200 0.1 (sm_100a)"; }

const char* cm_strerror(int code) {
  switch (code) {
    case CM_OK: return "ok";
    case CM_E_INVALID: return "invalid argument";
    case CM_E_CAPACITY: return "capacity exceeded";
    case CM_E_CUDA: return "CUDA error";
    case CM_E_NO_DEVICE: return "no usable CUDA device";
    case CM_E_KEY_RANGE: return "voxel grid exceeds the key range";
    case CM_E_INTERNAL: return "device watchdog tripped";
    case CM_E_NOT_READY: return "no cloud submitted";
    default: return "unknown error";
  }
}

const char* cm_last_error(cm_handle_t h) { return h ? h->last_error.c_str() : "null handle"; }

// ---- sensor_msgs/PointCloud2 adapters (pure host code) -------------------------------------------------------------------
int cm_layout_from_pointcloud2(const cm_pc2_field_t* fields, int n_fields, uint32_t point_step, int is_bigendian, int is_dense,
                               cm_layout_t* out) {
  if (!out || n_fields < 0 || (n_fields > 0 && !fields)) return CM_E_INVALID;
  if (is_bigendian) return CM_E_INVALID;  // the kernels read little-endian FLOAT32 (every ROS 1 driver on x86 / ARM emits that)
  if (point_step < 12 || point_step > 65535) return CM_E_INVALID;
  int32_t off[4] = {-1, -1, -1, -1};
  static const char* const kNames[4] = {"x", "y", "z", "intensity"};
  for (int f = 0; f < n_fields; ++f) {
    if (!fields[f].name) continue;
    for (int k = 0; k < 4; ++k) {
      if (strcmp(fields[f].name, kNames[k]) != 0 || off[k] >= 0) continue;
      // pcl::FieldMatches: same name, same datatype, same count (a count of 0 is read as 1)
      const bool match = fields[f].datatype == CM_PC2_FLOAT32 && (fields[f].count == 1 || fields[f].count == 0) &&
                         (uint64_t)fields[f].offset + 4u <= (uint64_t)point_step;
      if (match) off[k] = (int32_t)fields[f].offset;
      else if (k < 3) return CM_E_INVALID;  // PCL would leave the coordinate unset: refuse instead
    }
  }
  if (off[0] < 0 || off[1] < 0 || off[2] < 0) return CM_E_INVALID;
  out->point_step = (int32_t)point_step;
  out->off_x = off[0]; out->off_y = off[1]; out->off_z = off[2];
  out->off_intensity = off[3] >= 0 ? off[3] : CM_NO_FIELD;
  out->is_dense = is_dense ? 1 : 0;
  return CM_OK;
}

int cm_pointcloud2_describe(int out_point_step, int64_t n_points, cm_pc2_desc_t* out) {
  if (!out || (out_point_step != 16 && out_point_step != 32) || n_points < 0 || n_points > 0xFFFFFFFFll / out_point_step)
    return CM_E_INVALID;
  memset(out, 0, sizeof(*out));
  out->height = 1;                       // pcl::PassThrough / VoxelGrid / operator+= all leave height = 1, width = size
  out->width = (uint32_t)n_points;
  out->point_step = (uint32_t)out_point_step;
  out->row_step = (uint32_t)out_point_step * out->width;
  out->is_bigendian = 0;
  out->is_dense = 1;
  out->n_fields = 4;
  static const char* const kNames[4] = {"x", "y", "z", "intensity"};
  const uint32_t offs[4] = {0u, 4u, 8u, out_point_step == 32 ? 16u : 12u};  // pcl::PointXYZI: intensity behind the padded xyz1
  for (int k = 0; k < 4; ++k) {
    out->fields[k].name = kNames[k]; out->fields[k].offset = offs[k]; out->fields[k].datatype = CM_PC2_FLOAT32;
    out->fields[k].count = 1;
  }
  return CM_OK;
}

int cm_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int cm_create(const cm_config_t* cfg, cm_handle_t* out) {
  if (!cfg || !out) return CM_E_INVALID;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return CM_E_NO_DEVICE;
  if (cfg->device < 0 || cfg->device >= n) return CM_E_INVALID;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) return CM_E_CUDA;
  if (prop.major != 10) return CM_E_NO_DEVICE;  // sm_100a code only
  cm_handle_t h = new (std::nothrow) cm_handle_s();
  if (!h) return CM_E_INTERNAL;
  h->cfg = *cfg;
  cm_config_t& c = h->cfg;
  if (c.max_sensors <= 0) c.max_sensors = 6;
  if (c.max_sensors > CM_MAX_SENSORS) { delete h; return CM_E_INVALID; }
  if (c.max_points_per_sensor <= 0) c.max_points_per_sensor = 262144;
  if (c.max_point_step <= 0) c.max_point_step = 32;
  if (c.frames_in_flight <= 0) c.frames_in_flight = 2;
  if (c.frames_in_flight > 8) c.frames_in_flight = 8;
  if (c.max_batch_frames <= 0) c.max_batch_frames = 1;
  if (c.max_batch_points <= 0) c.max_batch_points = (int64_t)c.max_sensors * c.max_points_per_sensor * c.max_batch_frames;
  if (c.max_batch_segments <= 0) c.max_batch_segments = c.max_batch_frames * c.max_sensors;
  if (c.out_point_step != 32) c.out_point_step = 16;
  if (c.max_batch_points > 0xFFFFFFF0ll) { delete h; return CM_E_CAPACITY; }
  h->device = c.device;
  if (cudaSetDevice(h->device) != cudaSuccess) { delete h; return CM_E_CUDA; }
  if (configure_device_kernels() != cudaSuccess || configure_sort_kernels() != cudaSuccess ||
      configure_centroid_kernels() != cudaSuccess) {
    delete h;
    return CM_E_CUDA;
  }
  if (getenv("CM_NO_GRAPH")) h->use_graph = false;
  // debug: start the run epochs just below their wrap-around (k_grid_setup clears the look-back words and restarts at 16
  // once *epoch_dev + 64 reaches 2^30, about 67 M runs into the life of a handle), so that tests reach it
  if (const char* es = getenv("CM_EPOCH_START")) {
    char* end = nullptr;
    const unsigned long long v = strtoull(es, &end, 10);
    if (end == es || *end != '\0' || v % 16ull != 0ull || v >= (1ull << 30) - 64ull) { delete h; return CM_E_INVALID; }
    h->epoch_start = (uint32_t)v;
  }
  for (int s = 0; s < CM_MAX_SENSORS; ++s) {
    float* m = h->mats_host + s * 12;
    for (int k = 0; k < 12; ++k) m[k] = (k % 5 == 0) ? 1.f : 0.f;  // identity rows
  }
  // defaults = getROI with Parameter.h:31-35 (z [-0.5, 3], y +-5, x [-15, 60]) and Parameter.h:27-28 (0.1 m, 2 points)
  h->crop.n_pass = 3;
  h->crop.pass[0] = PassDev{2, -0.5f, 3.0f, 0};
  h->crop.pass[1] = PassDev{1, -10.0f / 2, 10.0f / 2, 0};
  h->crop.pass[2] = PassDev{0, -15.0f, 75.0f - 15.0f, 0};
  derive_box(h->crop);
  *out = h;
  return CM_OK;
}

int cm_destroy(cm_handle_t h) {
  if (!h) return CM_E_INVALID;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  delete h;
  return CM_OK;
}

int cm_set_extrinsic(cm_handle_t h, int sensor, const float* m16, int col_major) {
  if (!h || !m16) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (sensor < 0 || sensor >= h->cfg.max_sensors) return fail(h, CM_E_INVALID, "sensor %d out of range", sensor);
  float* m = h->mats_host + sensor * 12;
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 4; ++c) m[r * 4 + c] = col_major ? m16[c * 4 + r] : m16[r * 4 + c];
  return CM_OK;
}

int cm_set_extrinsic_tf(cm_handle_t h, int sensor, const double* q, const double* t) {
  if (!h || !q || !t) return CM_E_INVALID;
  // pcl_ros::transformPointCloud(in, out, tf::Transform): Eigen::Quaternionf(q.w, q.x, q.y, q.z), Vector3f(origin),
  // Affine3f(Translation3f(origin) * rotation); Eigen 3.3 QuaternionBase::toRotationMatrix.
  const float x = (float)q[0], y = (float)q[1], z = (float)q[2], w = (float)q[3];
  const float tx = 2.0f * x, ty = 2.0f * y, tz = 2.0f * z;
  const float twx = tx * w, twy = ty * w, twz = tz * w;
  const float txx = tx * x, txy = ty * x, txz = tz * x;
  const float tyy = ty * y, tyz = tz * y, tzz = tz * z;
  float m[16] = {1.0f - (tyy + tzz), txy - twz, txz + twy, (float)t[0],
                 txy + twz, 1.0f - (txx + tzz), tyz - twx, (float)t[1],
                 txz - twy, tyz + twx, 1.0f - (txx + tyy), (float)t[2],
                 0.f, 0.f, 0.f, 1.f};
  return cm_set_extrinsic(h, sensor, m, 0);
}

int cm_get_extrinsic(cm_handle_t h, int sensor, float* m12) {
  if (!h || !m12) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (sensor < 0 || sensor >= h->cfg.max_sensors) return fail(h, CM_E_INVALID, "sensor %d out of range", sensor);
  memcpy(m12, h->mats_host + sensor * 12, 12 * sizeof(float));
  return CM_OK;
}

int cm_set_crop(cm_handle_t h, int n_pass, const cm_pass_t* passes) {
  if (!h) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (n_pass < 0 || n_pass > CM_MAX_PASSES || (n_pass > 0 && !passes)) return fail(h, CM_E_INVALID, "0..%d passes", CM_MAX_PASSES);
  for (int k = 0; k < n_pass; ++k)
    if (passes[k].axis < 0 || passes[k].axis > 3) return fail(h, CM_E_INVALID, "pass %d: axis must be 0..3", k);
  h->crop.n_pass = n_pass;
  for (int k = 0; k < n_pass; ++k) h->crop.pass[k] = PassDev{passes[k].axis, passes[k].lo, passes[k].hi, passes[k].negative ? 1 : 0};
  derive_box(h->crop);
  return CM_OK;
}

namespace {
// Eigen 3.3 MatrixBase::isIdentity() with dummy_precision<float>() = 1e-5 on an Affine3f's matrix (its fourth row is exactly
// 0 0 0 1): relative on the diagonal (isApprox), absolute off it (isMuchSmallerThan).
bool eigen_is_identity(const float* m12) {
  const float prec = 1e-5f;
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 4; ++c) {
      const float v = m12[r * 4 + c];
      if (r == c ? !(std::fabs(v - 1.0f) <= std::min(std::fabs(v), 1.0f) * prec) : !(std::fabs(v) <= prec)) return false;
    }
  return true;
}

// What pcl::CropBox<PointT>::applyFilter (PCL 1.8.1) derives from its settings before the point loop, in float as it does.
void derive_obox(const cm_crop_box_t& b, OrientedBoxDev& d) {
  memset(&d, 0, sizeof(d));
  memcpy(d.t, b.transform, sizeof(d.t));
  memcpy(d.tr, b.translation, sizeof(d.tr));
  memcpy(d.mn, b.min, sizeof(d.mn));
  memcpy(d.mx, b.max, sizeof(d.mx));
  d.flags = b.negative ? OBOX_NEGATIVE : 0u;
  if (!eigen_is_identity(b.transform)) d.flags |= OBOX_TRANSFORM;
  if (b.translation[0] != 0.f || b.translation[1] != 0.f || b.translation[2] != 0.f) d.flags |= OBOX_TRANSLATE;
  const float roll = b.rotation[0], pitch = b.rotation[1], yaw = b.rotation[2];
  if (roll != 0.f || pitch != 0.f || yaw != 0.f) {
    // pcl::getTransformation(0, 0, 0, roll, pitch, yaw): float cos / sin
    const float A = std::cos(yaw), B = std::sin(yaw), C = std::cos(pitch), D = std::sin(pitch), E = std::cos(roll),
                F = std::sin(roll), DE = D * E, DF = D * F;
    const float m[3][3] = {{A * C, A * DF - B * E, B * F + A * DE}, {B * C, A * E + B * DF, B * DE - A * F}, {-D, C * F, C * E}};
    // Transform::inverse() (Affine): the linear part by Eigen's 3x3 cofactor inverse, then translation = -linear * (0, 0, 0)
    auto cof = [&](int i, int j) {
      const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
      return m[i1][j1] * m[i2][j2] - m[i1][j2] * m[i2][j1];
    };
    const float det = (cof(0, 0) * m[0][0] + cof(1, 0) * m[1][0]) + cof(2, 0) * m[2][0];
    const float invdet = 1.0f / det;
    for (int i = 0; i < 3; ++i) {
      for (int j = 0; j < 3; ++j) d.r[i * 4 + j] = cof(j, i) * invdet;
      d.r[i * 4 + 3] = ((-d.r[i * 4 + 0]) * 0.0f + (-d.r[i * 4 + 1]) * 0.0f) + (-d.r[i * 4 + 2]) * 0.0f;
    }
    if (!eigen_is_identity(d.r)) d.flags |= OBOX_ROTATE;
  }
}
}  // namespace

int cm_set_crop_boxes(cm_handle_t h, int n_boxes, const cm_crop_box_t* boxes) {
  if (!h) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (n_boxes < 0 || n_boxes > CM_MAX_CROP_BOXES || (n_boxes > 0 && !boxes))
    return fail(h, CM_E_INVALID, "0..%d crop boxes", CM_MAX_CROP_BOXES);
  for (int k = 0; k < n_boxes; ++k)
    for (int a = 0; a < 3; ++a)
      if (std::isnan(boxes[k].min[a]) || std::isnan(boxes[k].max[a])) return fail(h, CM_E_INVALID, "crop box %d: NaN limit", k);
  OrientedBoxDev d[CM_MAX_CROP_BOXES]{};
  for (int k = 0; k < n_boxes; ++k) derive_obox(boxes[k], d[k]);
  memcpy(h->obox, d, sizeof(d));
  h->n_obox = n_boxes;
  return CM_OK;
}

int cm_set_voxel(cm_handle_t h, const float* leaf3, int min_points, int downsample_all) {
  if (!h || !leaf3) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  for (int k = 0; k < 3; ++k)
    if (!(leaf3[k] > 0.f) || !std::isfinite(leaf3[k])) return fail(h, CM_E_INVALID, "leaf size must be positive");
  for (int k = 0; k < 3; ++k) {
    h->leaf[k] = leaf3[k];
    h->inv_leaf[k] = 1.0f / leaf3[k];  // PCL: inverse_leaf_size_ = Array4f::Ones() / leaf_size_.array()
  }
  h->min_points = min_points < 0 ? 0u : (uint32_t)min_points;
  h->downsample_all = downsample_all ? 1u : 0u;
  return CM_OK;
}

int cm_set_voxel_bounds(cm_handle_t h, const float* min3, const float* max3) {
  if (!h) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!min3 || !max3) { h->have_bounds = false; return CM_OK; }
  for (int k = 0; k < 3; ++k) {
    if (!std::isfinite(min3[k]) || !std::isfinite(max3[k]) || min3[k] > max3[k]) return fail(h, CM_E_INVALID, "bad bounds");
    h->bounds_min[k] = min3[k]; h->bounds_max[k] = max3[k];
  }
  h->have_bounds = true;
  return CM_OK;
}

int cm_set_overflow_mode(cm_handle_t h, int mode) {
  if (!h || (mode != 0 && mode != 1)) return CM_E_INVALID;
  h->overflow_mode = mode;
  return CM_OK;
}

int cm_set_submit_policy(cm_handle_t h, int policy) {
  if (!h || (policy != CM_SUBMIT_LATEST_WINS && policy != CM_SUBMIT_FIRST_WINS)) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  h->submit_policy = policy;
  return CM_OK;
}

int cm_set_profiling(cm_handle_t h, int on) {
  if (!h) return CM_E_INVALID;
  h->profiling = on != 0;
  return CM_OK;
}

int cm_submit_cloud(cm_handle_t h, int sensor, const void* data, int64_t n_points, const cm_layout_t* layout, uint64_t stamp) {
  return submit_impl(h, sensor, data, n_points, layout, stamp, false);
}

int cm_submit_cloud_pinned(cm_handle_t h, int sensor, const void* data, int64_t n_points, const cm_layout_t* layout,
                           uint64_t stamp) {
  return submit_impl(h, sensor, data, n_points, layout, stamp, true);
}

int cm_submit_clouds_pinned(cm_handle_t h, int count, const int* sensors, const void* const* data, const int64_t* n_points,
                            const cm_layout_t* layouts, const uint64_t* stamps) {
  if (!h || count < 0 || (count > 0 && (!sensors || !data || !n_points || !layouts))) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  int rc = ensure_host_path(h);
  if (rc != CM_OK) return rc;
  Slot& sl = h->slots[h->fill];
  if (sl.busy) return fail(h, CM_E_CAPACITY, "all %d frame slots are in flight: call cm_wait_frame first", h->cfg.frames_in_flight);
  for (int i = 0; i < count; ++i) {
    if (sensors[i] < 0 || sensors[i] >= h->cfg.max_sensors) return fail(h, CM_E_INVALID, "sensor %d out of range", sensors[i]);
    if (!layout_ok(layouts[i])) return fail(h, CM_E_INVALID, "cloud %d: bad layout", i);
    if (n_points[i] < 0 || (n_points[i] > 0 && !data[i])) return fail(h, CM_E_INVALID, "cloud %d: bad cloud", i);
    if (n_points[i] > h->cfg.max_points_per_sensor) return fail(h, CM_E_CAPACITY, "cloud %d: %lld points > max_points_per_sensor", i, (long long)n_points[i]);
    if (layouts[i].point_step > h->cfg.max_point_step) return fail(h, CM_E_CAPACITY, "cloud %d: point_step %d > max_point_step", i, layouts[i].point_step);
  }
  // Clouds that follow each other in host memory, belong to consecutive sensor ids and are 16-byte multiples travel as ONE
  // copy (a 2 MB copy reaches ~50 GB/s over PCIe 5 x16, an 8 MB one ~54) into the slot's frame arena: bump-allocated, so a
  // coalesced run never shares bytes with a sensor's own region (single submissions) or with another run. Superseded
  // clouds simply stay behind in the arena until the frame is merged; when it is full the clouds go one by one.
  std::vector<int> pick;
  pick.reserve((size_t)count);
  for (int i = 0; i < count; ++i) {
    if (h->submit_policy == CM_SUBMIT_FIRST_WINS && sl.sensor[sensors[i]].submitted) continue;  // the reference's flag gate
    pick.push_back(i);
  }
  size_t a = 0;
  while (a < pick.size()) {
    const int i = pick[a];
    size_t run_bytes = (size_t)n_points[i] * (size_t)layouts[i].point_step;
    size_t b = a + 1;
    while (b < pick.size() && pick[b] == pick[b - 1] + 1 && sensors[pick[b]] == sensors[pick[b - 1]] + 1 && run_bytes % 16 == 0 &&
           run_bytes > 0 && static_cast<const uint8_t*>(data[pick[b]]) == static_cast<const uint8_t*>(data[i]) + run_bytes) {
      run_bytes += (size_t)n_points[pick[b]] * (size_t)layouts[pick[b]].point_step;
      ++b;
    }
    const size_t need = align_up(run_bytes, kAlign);
    if (b - a >= 2 && sl.arena_used + need > sl.arena_bytes) b = a + 1;  // arena full: this cloud alone, into its own region
    cudaStream_t st = h->sensor_stream[sensors[i]].get();
    uint8_t* dst;
    if (b - a >= 2) {
      dst = sl.arena_dev.get() + sl.arena_used;
      sl.arena_used += need;
    } else {
      run_bytes = (size_t)n_points[i] * (size_t)layouts[i].point_step;
      dst = sl.raw_dev.get() + (size_t)sensors[i] * h->slot_stride;
    }
    if (run_bytes) CM_CUDA(h, cudaMemcpyAsync(dst, data[i], run_bytes, cudaMemcpyHostToDevice, st));
    size_t off = 0;
    for (size_t k = a; k < b; ++k) {
      const int c = pick[k];
      SensorState& ss = sl.sensor[sensors[c]];
      CM_CUDA(h, cudaEventRecord(ss.copied.get(), st));
      ss.submitted = true; ss.n_points = n_points[c]; ss.layout = layouts[c]; ss.stamp = stamps ? stamps[c] : 0;
      ss.dev = dst + off;
      off += (size_t)n_points[c] * (size_t)layouts[c].point_step;
    }
    a = b;
  }
  return CM_OK;
}

int cm_merge_frame_async(cm_handle_t h, uint64_t sensor_mask, int64_t* ticket) {
  if (!h || !ticket) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  return merge_async_impl(h, sensor_mask, ticket);
}

int cm_wait_frame(cm_handle_t h, int64_t ticket, cm_frame_out_t* out, uint64_t* out_used_mask, uint64_t* out_stamp) {
  if (!h) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  return wait_impl(h, ticket, out, out_used_mask, out_stamp);
}

int cm_wait_frame_view(cm_handle_t h, int64_t ticket, cm_frame_view_t* view) {
  if (!h || !view) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  Slot* sl = nullptr;
  for (auto& s : h->slots) if (s.busy && s.ticket == ticket) sl = &s;
  if (!sl) return fail(h, CM_E_INVALID, "unknown ticket %lld", (long long)ticket);
  uint64_t used = 0, stamp = 0;
  int rc = wait_impl(h, ticket, nullptr, &used, &stamp);  // one synchronisation; nothing is copied
  if (rc != CM_OK) return rc;
  const cm_frame_info_t& fi = h->frame_info[0];
  memset(view, 0, sizeof(*view));
  view->info = fi;
  view->n_survivors = fi.survivor_end - fi.survivor_begin;
  view->n_voxels = fi.voxel_end - fi.voxel_begin;
  view->used_mask = used; view->stamp = stamp;
  if (h->overflow_mode == 1 && fi.pcl_overflow)
    return fail(h, CM_E_INVALID, "PCL would refuse this frame (leaf too small): its result is the merged cloud, use cm_wait_frame");
  if ((uint64_t)view->n_voxels > sl->exp_cap) return fail(h, CM_E_CAPACITY, "more voxels than the result mirror holds");
  view->voxel_xyzi = sl->exp_xyzi.get();
  view->voxel_count = sl->exp_count.get();
  view->voxel_idx = reinterpret_cast<const uint64_t*>(sl->exp_idx.get());
  return CM_OK;
}

int cm_merge_frame(cm_handle_t h, uint64_t sensor_mask, cm_frame_out_t* out, uint64_t* out_used_mask, uint64_t* out_stamp) {
  if (!h) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  int64_t ticket = 0;
  int rc = merge_async_impl(h, sensor_mask, &ticket);
  if (rc != CM_OK) return rc;
  return wait_impl(h, ticket, out, out_used_mask, out_stamp);
}

int cm_host_alloc(void** p, size_t bytes) {
  if (!p) return CM_E_INVALID;
  HostPtr<void> mem;
  const cudaError_t e = pinned_alloc(mem, bytes, cudaHostAllocDefault);
  *p = mem.release();  // the caller's from here on (cm_host_free)
  return e == cudaSuccess ? CM_OK : CM_E_CUDA;
}
int cm_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? CM_OK : CM_E_CUDA; }

int cm_run_batch(cm_handle_t h, const cm_segment_t* segments, int n_segments, void* stream) {
  if (!h) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  int rc = ensure_batch_ws(h);
  if (rc != CM_OK) return rc;
  return run_pipeline(h, h->batch, segments, n_segments, static_cast<cudaStream_t>(stream), true);
}

int cm_dev_transform_crop(cm_handle_t h, const cm_segment_t* segments, int n_segments, void* stream) {
  if (!h) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  int rc = ensure_batch_ws(h);
  if (rc != CM_OK) return rc;
  return run_pipeline(h, h->batch, segments, n_segments, static_cast<cudaStream_t>(stream), false);
}

namespace {
// The cloud of a cm_dev_* entry point: n_points packed float4 in device memory.
int check_dev_cloud(cm_handle_t h, const void* xyzi_dev, int64_t n_points) {
  if (n_points > 0 && (!xyzi_dev || (reinterpret_cast<uintptr_t>(xyzi_dev) & 15u)))
    return fail(h, CM_E_INVALID, "the device cloud must be a 16-byte aligned pointer");
  if (n_points < 0) return fail(h, CM_E_INVALID, "bad n_points");
  return CM_OK;
}

// VoxelGrid of n packed points on the batch workspace. seed_enc_dev: device-resident bounds (GiantPlan::enc) folded into the
// local box; known_idx_bits >= 0: the key plan is known on the host, no device round trip.
int voxelgrid_run(cm_handle_t h, const float4* pts, int64_t n_points, cudaStream_t st, const uint32_t* seed_enc_dev = nullptr,
                  int known_idx_bits = -1) {
  int rc = ensure_batch_ws(h);
  if (rc != CM_OK) return rc;
  Workspace& w = h->batch;
  if (n_points < 0 || n_points > (int64_t)w.cap_points) return fail(h, CM_E_CAPACITY, "%lld points > capacity %u", (long long)n_points, w.cap_points);
  w.has_run = true; w.report_valid = false; w.profiled = h->profiling;
  w.n_frames = 1; w.n_segs = 0; w.points_in = n_points; w.launches = 0;
  w.ran_k1 = false; w.ran_voxel = false; w.stream = st; w.n_k1_tiles = 0; w.dense_valid = false;
  w.voxel_pts = pts; w.fused_keys = false;
  h->last = &w;
  CM_CUDA(h, cudaEventRecord(w.ev[EV_START].get(), st));
  CM_CUDA(h, cudaMemsetAsync(w.meta.get(), 0, w.ml.zero_bytes, st));
  VoxelParams vp;
  fill_voxel_params(h, w, vp, w.voxel_pts, 1, (uint32_t)n_points);
  CM_CUDA(h, launch_minmax(w.voxel_pts, (uint32_t)n_points, vp.ctrl, vp.acc, const_cast<uint32_t*>(vp.frame_surv_start), st));
  ++w.launches;
  if (seed_enc_dev) {
    CM_CUDA(h, launch_seed_bounds_enc(vp.acc, seed_enc_dev, st));
    ++w.launches;
  } else if (h->have_bounds) {
    CM_CUDA(h, launch_seed_bounds(vp.acc, h->bounds_min, h->bounds_max, st));
    ++w.launches;
  }
  CM_CUDA(h, cudaEventRecord(w.ev[EV_K1].get(), st));
  return run_voxel(h, w, vp, st, false, true, known_idx_bits);
}
}  // namespace

int cm_dev_voxelgrid(cm_handle_t h, const float* xyzi_dev, int64_t n_points, int is_dense, void* stream) {
  (void)is_dense;  // non-finite points are skipped either way (PCL skips them when !is_dense; undefined otherwise)
  if (!h) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  const int rc = check_dev_cloud(h, xyzi_dev, n_points);
  if (rc != CM_OK) return rc;
  return voxelgrid_run(h, reinterpret_cast<const float4*>(xyzi_dev), n_points, static_cast<cudaStream_t>(stream));
}

// ---- zone slicing ---------------------------------------------------------------------------------------------------------
namespace {
// The device form of n_zones PassThrough chains, each with its box form where the chain allows it (see ZoneDev).
int make_zone_set(cm_handle_t h, int n_zones, const cm_zone_t* zones, ZoneSet& zs) {
  zs = ZoneSet{};
  zs.n_zones = n_zones;
  zs.all_box = n_zones > 0 ? 1 : 0;
  for (int z = 0; z < n_zones; ++z) {
    if (zones[z].n_pass < 0 || zones[z].n_pass > CM_MAX_ZONE_PASSES) return fail(h, CM_E_INVALID, "zone %d: bad n_pass", z);
    ZoneDev& zd = zs.zone[z];
    zd.n_pass = zones[z].n_pass;
    for (int k = 0; k < zones[z].n_pass; ++k) {
      const cm_pass_t& ps = zones[z].pass[k];
      if (ps.axis < 0 || ps.axis > 3) return fail(h, CM_E_INVALID, "zone %d pass %d: bad axis", z, k);
      zd.pass[k] = PassDev{ps.axis, ps.lo, ps.hi, ps.negative ? 1 : 0};
    }
    derive_box(zd);
    if (!zd.is_box) zs.all_box = 0;
  }
  return CM_OK;
}
}  // namespace

int cm_set_zones(cm_handle_t h, int n_zones, const cm_zone_t* zones) {
  if (!h || n_zones < 0 || n_zones > CM_MAX_ZONES || (n_zones > 0 && !zones)) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  ZoneSet zs;
  const int rc = make_zone_set(h, n_zones, zones, zs);
  if (rc == CM_OK) h->zones = zs;
  return rc;
}

namespace {
// capacity: the input may hold up to `points`; the zones together up to twice that (boundary duplicates are rare, but
// zones are free to overlap)
int zone_ws_ensure(cm_handle_t h, size_t points) {
  cm_handle_s::ZoneWs& z = h->zw;
  const size_t want = std::max<size_t>({points, (size_t)h->cfg.max_batch_points, (size_t)1});
  if (z.cap_points >= want) return CM_OK;
  z = cm_handle_s::ZoneWs();  // the old buffers go before the larger ones are allocated
  const size_t tiles = want / zone_tile_points() + 2;
  CM_CUDA(h, dev_alloc(z.mask, want));
  CM_CUDA(h, dev_alloc(z.tile_count, tiles * CM_MAX_ZONES));
  CM_CUDA(h, dev_alloc(z.tile_offset, tiles * CM_MAX_ZONES));
  CM_CUDA(h, dev_alloc(z.zone_begin, (size_t)CM_MAX_ZONES + 2));
  CM_CUDA(h, dev_alloc(z.overflow, (size_t)1));
  CM_CUDA(h, dev_alloc(z.zone_total, (size_t)CM_MAX_ZONES + 2));
  CM_CUDA(h, cudaMemset(z.zone_total.get(), 0, sizeof(uint32_t) * (CM_MAX_ZONES + 2)));
  z.cap_out = 2 * want;
  CM_CUDA(h, dev_alloc(z.out_xyzi, z.cap_out));
  CM_CUDA(h, dev_alloc(z.out_src, z.cap_out));
  CM_CUDA(h, pinned_alloc(z.report, sizeof(uint32_t) * (CM_MAX_ZONES + 3), cudaHostAllocDefault));
  CM_CUDA(h, cudaDeviceSynchronize());  // the clear above ran on the default stream (see ws_alloc)
  z.cap_points = want;
  return CM_OK;
}

// A stage writes its results into the handle's zone outputs: an input that lives there would be overwritten while it is
// still being read (chain stages over separate handles, or copy the cloud out first).
bool in_zone_outputs(cm_handle_t h, const void* p, int64_t n_points) {
  const cm_handle_s::ZoneWs& z = h->zw;
  if (!p || !z.out_xyzi || n_points <= 0) return false;
  const uintptr_t a = reinterpret_cast<uintptr_t>(p), b = a + (uintptr_t)n_points * 16u;
  const uintptr_t lo = reinterpret_cast<uintptr_t>(z.out_xyzi.get()), hi = lo + (uintptr_t)z.cap_out * 16u;
  return a < hi && b > lo;
}

// The clouds [begin[k], begin[k+1]) of pts that a multi-cloud filter takes.
int check_clouds(cm_handle_t h, const float4* pts, const int64_t* begin, int n_clouds, int max_clouds) {
  if (n_clouds < 1 || n_clouds > max_clouds) return fail(h, CM_E_INVALID, "1 .. %d clouds per call", max_clouds);
  if (begin[0] != 0) return fail(h, CM_E_INVALID, "begin[0] must be 0");
  for (int c = 0; c < n_clouds; ++c)
    if (begin[c + 1] < begin[c]) return fail(h, CM_E_INVALID, "begin must not decrease");
  const int rc = check_dev_cloud(h, pts, begin[n_clouds]);
  if (rc != CM_OK) return rc;
  if (in_zone_outputs(h, pts, begin[n_clouds]))
    return fail(h, CM_E_INVALID, "the input cloud lies in this handle's own zone outputs (use another handle or copy it out)");
  return CM_OK;
}

// the launch parameters of one split of `pts` over the handle's zone workspace (which must hold n_points)
ZoneParams zone_params(cm_handle_t h, const float4* pts, int64_t n_points, bool mask_given, int given_zones) {
  cm_handle_s::ZoneWs& z = h->zw;
  ZoneParams zp;
  zp.pts = pts; zp.n_points = (uint32_t)n_points;
  zp.n_tiles = (uint32_t)((n_points + zone_tile_points() - 1) / zone_tile_points());
  zp.zones = h->zones;
  zp.mask_given = mask_given ? 1u : 0u;
  if (mask_given) {  // one output: the points whose flag is set
    zp.zones = ZoneSet{};
    zp.zones.n_zones = given_zones;
  }
  z.n_zones_run = zp.zones.n_zones;
  zp.mask = z.mask.get(); zp.tile_count = z.tile_count.get(); zp.tile_offset = z.tile_offset.get(); zp.zone_begin = z.zone_begin.get();
  zp.zone_total = z.zone_total.get(); zp.scan_ticket = z.zone_total.get() + CM_MAX_ZONES;
  zp.overflow = z.overflow.get(); zp.out_capacity = (uint32_t)std::min<size_t>(z.cap_out, 0xFFFFFFF0u);
  zp.out_xyzi = z.out_xyzi.get(); zp.out_src = z.out_src.get();
  for (int i = 0; i < CM_MAX_ZONES; ++i) zp.zone_ptr[i] = nullptr;
  zp.zone_remote_base = nullptr;
  zp.giant_plan = nullptr; zp.giant_invalid_part = 0;
  return zp;
}

// giant != null: the zones are the given_zones ranks of the giant-cloud mode and the masks come from the device-resident plan
int zone_run(cm_handle_t h, const float4* pts, int64_t n_points, cudaStream_t st, bool mask_given = false,
             int given_zones = 1, const GiantPlan* giant = nullptr, uint32_t giant_invalid_part = 0) {
  cm_handle_s::ZoneWs& z = h->zw;
  if (!mask_given && h->zones.n_zones <= 0) return fail(h, CM_E_INVALID, "no zones configured (cm_set_zones)");
  if (n_points < 0 || n_points > 0xFFFFFFF0ll) return fail(h, CM_E_INVALID, "bad n_points");
  if (in_zone_outputs(h, pts, n_points))
    return fail(h, CM_E_INVALID, "the input cloud lies in this handle's own zone outputs (use another handle or copy it out)");
  int rc = zone_ws_ensure(h, (size_t)n_points);
  if (rc != CM_OK) return rc;
  ZoneParams zp = zone_params(h, pts, n_points, mask_given, given_zones);
  if (giant) { zp.mask_given = 0; zp.giant_plan = giant; zp.giant_invalid_part = giant_invalid_part; }
  CM_CUDA(h, cudaMemsetAsync(z.overflow.get(), 0, sizeof(uint32_t), st));
  CM_CUDA(h, launch_zone_split(zp, st));
  CM_CUDA(h, cudaMemcpyAsync(z.report.get(), z.zone_begin.get(), sizeof(uint32_t) * (CM_MAX_ZONES + 1), cudaMemcpyDeviceToHost, st));
  CM_CUDA(h, cudaMemcpyAsync(z.report.get() + CM_MAX_ZONES + 1, z.overflow.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  z.stream = st; z.ran = true; z.launches = zp.n_tiles ? CM_ZONE_LAUNCHES : 1; z.last = zp; z.ror_run = false;
  return CM_OK;
}
}  // namespace

int cm_dev_zone_split(cm_handle_t h, const float* xyzi_dev, int64_t n_points, void* stream) {
  if (!h) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (xyzi_dev) {
    const int rc = check_dev_cloud(h, xyzi_dev, n_points);
    return rc == CM_OK ? zone_run(h, reinterpret_cast<const float4*>(xyzi_dev), n_points, st) : rc;
  }
  // the merged cropped cloud of the last transform_crop run (what getROI hands to getCloudPart)
  if (!h->last || !h->last->ran_k1) return fail(h, CM_E_INVALID, "no transform_crop result on this handle");
  Workspace& w = *h->last;
  int rc = fetch_report(h, w);
  if (rc != CM_OK) return rc;
  rc = materialize_dense(h, w);
  if (rc != CM_OK) return rc;
  CM_CUDA(h, cudaStreamSynchronize(w.stream));
  return zone_run(h, w.dense_xyzi.get(), h->stats.survivors, st);
}

namespace {
int zone_out_locked(cm_handle_t h, cm_zone_out_t* out);
}
int cm_get_zone_out(cm_handle_t h, cm_zone_out_t* out) {
  if (!h || !out) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  return zone_out_locked(h, out);
}
namespace {
int zone_out_locked(cm_handle_t h, cm_zone_out_t* out) {
  cm_handle_s::ZoneWs& z = h->zw;
  if (!z.ran) return fail(h, CM_E_INVALID, "no zone split has run on this handle");
  CM_CUDA(h, cudaSetDevice(h->device));
  CM_CUDA(h, cudaStreamSynchronize(z.stream));
  uint32_t* report = z.report.get();
  if (report[CM_MAX_ZONES + 1] && (size_t)report[CM_MAX_ZONES + 1] <= 0xFFFFFFF0u) {
    // Overlapping zones hold more points together than the output arrays were sized for (twice the input): grow them to
    // the size the scan found and repeat the scatter. The input cloud must still be where it was.
    const size_t need = report[CM_MAX_ZONES + 1];
    z.out_xyzi.reset(); z.out_src.reset(); z.cap_out = 0;  // the old outputs go before the larger ones are allocated
    CM_CUDA(h, dev_alloc(z.out_xyzi, need));
    CM_CUDA(h, dev_alloc(z.out_src, need));
    z.cap_out = need;
    z.last.out_xyzi = z.out_xyzi.get(); z.last.out_src = z.out_src.get(); z.last.out_capacity = (uint32_t)need;
    CM_CUDA(h, cudaMemsetAsync(z.overflow.get(), 0, sizeof(uint32_t), z.stream));
    CM_CUDA(h, launch_zone_scatter(z.last, z.stream));
    CM_CUDA(h, cudaStreamSynchronize(z.stream));
    report[CM_MAX_ZONES + 1] = 0;
    ++z.launches;
  }
  memset(out, 0, sizeof(*out));
  out->n_zones = z.n_zones_run;
  for (int k = 0; k <= z.n_zones_run; ++k) out->begin[k] = report[k];
  out->xyzi = reinterpret_cast<const float*>(z.out_xyzi.get());
  out->src = z.out_src.get();
  if (report[CM_MAX_ZONES + 1])
    return fail(h, CM_E_CAPACITY, "the zones hold %u points together, capacity is %zu", report[CM_MAX_ZONES + 1], z.cap_out);
  if (z.ror_run && report[CM_MAX_ZONES + 2] == CM_DEV_E_KEY_RANGE)
    return fail(h, CM_E_KEY_RANGE, "radius too small for the extent of a cloud (more than 2^14 cells from the origin)");
  if (z.ror_run && report[CM_MAX_ZONES + 2]) return fail(h, CM_E_INTERNAL, "device error %u", report[CM_MAX_ZONES + 2]);
  return CM_OK;
}

// The host-buffer forms: the caller's cloud is uploaded on the legacy stream into the handle's staging buffer.
int stage_host_cloud(cm_handle_t h, const float* xyzi_host, int64_t n_points, const float4** staged) {
  if (n_points < 0 || (n_points > 0 && !xyzi_host)) return fail(h, CM_E_INVALID, "bad host cloud");
  if (h->stage_cap < (size_t)n_points || !h->stage) {
    const size_t want = std::max<size_t>({(size_t)n_points, (size_t)h->cfg.max_batch_points, (size_t)1});
    h->stage.reset(); h->stage_cap = 0;  // the old buffer goes before the larger one is allocated
    CM_CUDA(h, dev_alloc(h->stage, want));
    h->stage_cap = want;
  }
  if (n_points) CM_CUDA(h, cudaMemcpyAsync(h->stage.get(), xyzi_host, (size_t)n_points * 16, cudaMemcpyHostToDevice, nullptr));
  *staged = h->stage.get();
  return CM_OK;
}

// ... and the zone outputs come back: the first n_offsets offsets of the report (zeros if it was never filled) into
// out_begin, then the points, or CM_E_CAPACITY (the needed size in out_begin[n_offsets - 1]) when they do not fit.
int zone_copy_out(cm_handle_t h, int n_offsets, float* out_xyzi, uint32_t* out_idx, int64_t capacity, int64_t* out_begin) {
  cm_zone_out_t zo{};
  const int rc = zone_out_locked(h, &zo);
  for (int k = 0; k < n_offsets; ++k) out_begin[k] = zo.begin[k];
  if (rc != CM_OK) return rc;
  const int64_t total = zo.begin[n_offsets - 1];
  if (total > capacity) return fail(h, CM_E_CAPACITY, "%lld points, caller capacity %lld", (long long)total, (long long)capacity);
  if (out_xyzi && total) CM_CUDA(h, cudaMemcpy(out_xyzi, zo.xyzi, (size_t)total * 16, cudaMemcpyDeviceToHost));
  if (out_idx && total) CM_CUDA(h, cudaMemcpy(out_idx, zo.src, (size_t)total * 4, cudaMemcpyDeviceToHost));
  return CM_OK;
}
}  // namespace

int cm_zone_split(cm_handle_t h, const float* xyzi_host, int64_t n_points, float* out_xyzi, uint32_t* out_src,
                  int64_t capacity, int64_t* out_begin) {
  if (!h || !out_begin || n_points < 0 || (n_points > 0 && !xyzi_host)) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  const float4* pts = nullptr;
  int rc = stage_host_cloud(h, xyzi_host, n_points, &pts);
  if (rc == CM_OK) rc = zone_run(h, pts, n_points, nullptr);
  return rc == CM_OK ? zone_copy_out(h, h->zones.n_zones + 1, out_xyzi, out_src, capacity, out_begin) : rc;
}

// ---- giant-cloud mode: bounding box, key histogram, routing by key range ------------------------------------------------
namespace {
// PCL's grid (VoxelGrid::applyFilter, float32) on a bounding box, with the handle's leaf
int route_grid(cm_handle_t h, const float* min3, const float* max3, RouteGrid* g, unsigned long long* cells) {
  long long div[3];
  for (int k = 0; k < 3; ++k) {
    g->inv[k] = h->inv_leaf[k];
    const float fmn = std::floor(min3[k] * h->inv_leaf[k]), fmx = std::floor(max3[k] * h->inv_leaf[k]);
    if (!(std::fabs(fmn) < 1073741824.f) || !(std::fabs(fmx) < 1073741824.f) || fmx < fmn)
      return fail(h, CM_E_KEY_RANGE, "bounding box outside the key range");
    g->min_b[k] = (long long)fmn;
    div[k] = (long long)fmx - (long long)fmn + 1;
    if (div[k] > (1ll << 21)) return fail(h, CM_E_KEY_RANGE, "more than 2^21 cells on an axis");
  }
  g->div0 = div[0];
  g->div01 = div[0] * div[1];
  if (cells) *cells = (unsigned long long)div[0] * (unsigned long long)div[1] * (unsigned long long)div[2];
  return CM_OK;
}
}  // namespace

int cm_dev_bounds(cm_handle_t h, const float* xyzi_dev, int64_t n_points, float* min3, float* max3, int64_t* n_finite,
                  void* stream) {
  if (!h || !min3 || !max3 || n_points < 0 || n_points > 0xFFFFFFF0ll) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  int rc = ensure_batch_ws(h);
  if (rc != CM_OK) return rc;
  Workspace& w = h->batch;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CM_CUDA(h, cudaMemsetAsync(w.meta.get(), 0, w.ml.zero_bytes, st));
  Ctrl* ctrl = reinterpret_cast<Ctrl*>(w.meta.get() + w.ml.off_ctrl);
  FrameAcc* acc = reinterpret_cast<FrameAcc*>(w.meta.get() + w.ml.off_acc);
  CM_CUDA(h, launch_minmax(reinterpret_cast<const float4*>(xyzi_dev), (uint32_t)n_points, ctrl, acc,
                           reinterpret_cast<uint32_t*>(w.meta.get() + w.ml.off_fstart), st));
  FrameAcc a;
  CM_CUDA(h, cudaMemcpyAsync(&a, acc, sizeof(a), cudaMemcpyDeviceToHost, st));
  CM_CUDA(h, cudaStreamSynchronize(st));
  const bool empty = a.max_enc[0] == 0u && a.nmin_enc[0] == 0u;
  for (int k = 0; k < 3; ++k) {
    uint32_t lo = f32_order_dec(~a.nmin_enc[k]), hi = f32_order_dec(a.max_enc[k]);
    float flo, fhi;
    memcpy(&flo, &lo, 4); memcpy(&fhi, &hi, 4);
    min3[k] = empty ? std::numeric_limits<float>::max() : flo;
    max3[k] = empty ? -std::numeric_limits<float>::max() : fhi;
  }
  if (n_finite) *n_finite = n_points - (int64_t)a.n_invalid;
  return CM_OK;
}

int cm_dev_key_histogram(cm_handle_t h, const float* xyzi_dev, int64_t n_points, const float* min3, const float* max3,
                         int bins, uint64_t* hist_dev, uint64_t* out_bin_width, void* stream) {
  if (!h || !min3 || !max3 || !hist_dev || bins <= 0 || n_points < 0 || n_points > 0xFFFFFFF0ll) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  RouteGrid g;
  unsigned long long cells = 0;
  int rc = route_grid(h, min3, max3, &g, &cells);
  if (rc != CM_OK) return rc;
  const unsigned long long width = std::max<unsigned long long>(1ull, (cells + (unsigned long long)bins - 1ull) / (unsigned long long)bins);
  if (out_bin_width) *out_bin_width = width;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CM_CUDA(h, cudaMemsetAsync(hist_dev, 0, sizeof(uint64_t) * (size_t)bins, st));
  CM_CUDA(h, launch_route_hist(reinterpret_cast<const float4*>(xyzi_dev), (uint32_t)n_points, g, width, (uint32_t)bins,
                               reinterpret_cast<unsigned long long*>(hist_dev), st));
  return CM_OK;
}

int cm_dev_route_by_key(cm_handle_t h, const float* xyzi_dev, int64_t n_points, const float* min3, const float* max3,
                        const uint64_t* splitters, int n_parts, int invalid_part, void* stream) {
  if (!h || !min3 || !max3 || n_parts < 1 || n_parts > CM_MAX_ZONES || (n_parts > 1 && !splitters) || invalid_part < 0 ||
      invalid_part >= n_parts || n_points < 0 || n_points > 0xFFFFFFF0ll)
    return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  int rc = check_dev_cloud(h, xyzi_dev, n_points);
  if (rc != CM_OK) return rc;
  RouteGrid g;
  rc = route_grid(h, min3, max3, &g, nullptr);
  if (rc != CM_OK) return rc;
  rc = zone_ws_ensure(h, (size_t)n_points);
  if (rc != CM_OK) return rc;
  RouteSplit sp{};
  sp.n_parts = n_parts; sp.invalid_part = (uint32_t)invalid_part;
  for (int k = 0; k + 1 < n_parts; ++k) sp.splitter[k] = splitters[k];
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CM_CUDA(h, launch_route_mask(reinterpret_cast<const float4*>(xyzi_dev), (uint32_t)n_points, g, sp, h->zw.mask.get(), st));
  return zone_run(h, reinterpret_cast<const float4*>(xyzi_dev), n_points, st, true, n_parts);
}

int cm_memcpy_d2d(cm_handle_t h, void* dst_dev, const void* src_dev, size_t bytes, void* stream) {
  if (!h) return CM_E_INVALID;
  CM_CUDA(h, cudaSetDevice(h->device));
  if (bytes) CM_CUDA(h, cudaMemcpyAsync(dst_dev, src_dev, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return CM_OK;
}

// ---- the cell-key front end of the outlier removals ----------------------------------------------------------------------
// Both removals search neighbours on the points sorted by cell key, clouds = the ranges [begin[k], begin[k+1]) of pts as
// the frames of the key (no neighbours across clouds), on the batch workspace. The statistical removal picks its cell edge
// from the bounds, so the front end is three steps: the bounds, the keys and sort on a given cell grid, the cell table.
namespace {
// Bounding box and non-finite count of every cloud (FrameAcc), and the cloud starts.
int cell_keys_begin(cm_handle_t h, const float4* pts, const int64_t* begin, int n_clouds, VoxelParams& vp, cudaStream_t st) {
  const int64_t n_points = begin[n_clouds];
  int rc = ensure_batch_ws(h);
  if (rc != CM_OK) return rc;
  Workspace& w = h->batch;
  if (n_points > (int64_t)w.cap_points) return fail(h, CM_E_CAPACITY, "%lld points > capacity %u", (long long)n_points, w.cap_points);
  if ((uint32_t)n_clouds > w.cap_frames)
    return fail(h, CM_E_CAPACITY, "%d clouds > max_batch_frames %u of this handle", n_clouds, w.cap_frames);
  rc = zone_ws_ensure(h, (size_t)n_points);
  if (rc != CM_OK) return rc;
  w.has_run = true; w.report_valid = false; w.profiled = false;
  w.n_frames = (uint32_t)n_clouds; w.n_segs = 0; w.points_in = n_points; w.launches = 0;
  w.ran_k1 = false; w.ran_voxel = false; w.stream = st; w.n_k1_tiles = 0; w.dense_valid = false;
  w.voxel_pts = pts; w.fused_keys = false;
  h->last = &w;
  CM_CUDA(h, cudaEventRecord(w.ev[EV_START].get(), st));
  CM_CUDA(h, cudaMemsetAsync(w.meta.get(), 0, w.ml.zero_bytes, st));
  fill_voxel_params(h, w, vp, pts, (uint32_t)n_clouds, (uint32_t)n_points);
  vp.pcl_refuses = 0;  // a cell grid of the neighbour search beyond the key range is always an error
  uint32_t* fss = const_cast<uint32_t*>(vp.frame_surv_start);
  for (int c = 0; c < n_clouds; ++c) {  // bounding box of every cloud (its own cell grid)
    const uint32_t n_here = (uint32_t)(begin[c + 1] - begin[c]);
    if (!n_here) continue;
    CM_CUDA(h, launch_minmax(pts + begin[c], n_here, vp.ctrl, vp.acc + c, fss + c, st));
    ++w.launches;
  }
  if (n_clouds > 1 || n_points == 0) {  // the cloud ranges (the single-cloud launch above wrote them itself)
    uint32_t starts[CM_MAX_ZONES + 1];
    for (int c = 0; c <= n_clouds; ++c) starts[c] = (uint32_t)begin[c];
    CM_CUDA(h, cudaMemcpyAsync(fss, starts, sizeof(uint32_t) * (size_t)(n_clouds + 1), cudaMemcpyHostToDevice, st));
  }
  return CM_OK;
}

// Cell keys of edge 1 / inv and their sort (no centroids).
int cell_keys_sort(cm_handle_t h, VoxelParams& vp, float inv, cudaStream_t st) {
  Workspace& w = h->batch;
  for (int k = 0; k < 3; ++k) vp.inv_leaf[k] = inv;
  CM_CUDA(h, cudaEventRecord(w.ev[EV_K1].get(), st));
  int rc = run_voxel(h, w, vp, st, false, false);  // keys + sort only
  if (rc != CM_OK) return rc;
  // A cloud whose grid k_grid_setup could not key (more than 2^21 cells on an axis, a coordinate beyond 2^30 cells) has
  // all its keys at 0 but keeps its real div_b: the cell table would be sized without it and the row walk would leave it.
  // The plan fetch above brought the verdict along, so such a call stops here, before the table and the search.
  if (w.plan_error == CM_DEV_E_KEY_RANGE) return fail(h, CM_E_KEY_RANGE, "cell too small for the extent of a cloud (cell grid exceeds the key range)");
  if (w.plan_error) return fail(h, CM_E_INTERNAL, "device error %u", w.plan_error);
  vp.key_bytes = w.key_bytes;
  return CM_OK;
}

// A small key space (the usual case: a cropped cloud) gets a direct-address table of the cells' first sorted positions
// instead of binary searches per point: rp.cell_start, else nullptr. no_table_env names the removal's test hook that forces
// the binary searches (the large-key-space path).
int enqueue_cell_table(cm_handle_t h, const VoxelParams& vp, const char* no_table_env, RorParams& rp, cudaStream_t st) {
  Workspace& w = h->batch;
  const uint32_t n_clouds = vp.n_frames;
  rp.cell_start = nullptr; rp.table_keys = 0;
  if (vp.max_points > 0 && w.plan_idx_bits <= 25 && ((uint64_t)n_clouds << w.plan_idx_bits) <= (1ull << 25) &&
      !getenv(no_table_env)) {
    const size_t keys = (size_t)n_clouds << w.plan_idx_bits;
    if (h->cell_table_cap < keys + 1) {
      h->cell_table.reset(); h->cell_table_cap = 0;  // the old table goes before the larger one is allocated
      CM_CUDA(h, dev_alloc(h->cell_table, keys + 1));
      h->cell_table_cap = keys + 1;
    }
    rp.cell_start = h->cell_table.get(); rp.table_keys = (uint32_t)keys;
    CM_CUDA(h, launch_radius_table(vp, rp, st));
    ++w.launches;
  }
  return CM_OK;
}
}  // namespace

// ---- radius outlier removal ---------------------------------------------------------------------------------------------
namespace {
// output zone k = the survivors of cloud k
int radius_outlier_run(cm_handle_t h, const float4* pts, const int64_t* begin, int n_clouds, double radius, int min_neighbors,
                       int negative, cudaStream_t st) {
  if (!(radius > 0.0) || min_neighbors < 0) return fail(h, CM_E_INVALID, "radius must be > 0 and min_neighbors >= 0");
  int rc = check_clouds(h, pts, begin, n_clouds, CM_MAX_ZONES);
  if (rc != CM_OK) return rc;
  const int64_t n_points = begin[n_clouds];
  VoxelParams vp;
  rc = cell_keys_begin(h, pts, begin, n_clouds, vp, st);
  if (rc != CM_OK) return rc;
  // cells a little wider than the radius: two points closer than the radius are then at most one cell apart on every
  // axis even after the float rounding of x * (1 / cell) (valid below 2^14 cells from the origin, checked on the device)
  const float cell = (float)radius * 1.00390625f;
  rc = cell_keys_sort(h, vp, 1.0f / cell, st);
  if (rc != CM_OK) return rc;
  Workspace& w = h->batch;
  RorParams rp;
  rp.r2 = (float)(radius * radius);
  rp.min_pts = (uint32_t)min_neighbors;
  rp.negative = negative ? 1u : 0u;
  rp.mask = h->zw.mask.get();
  rc = enqueue_cell_table(h, vp, "CM_ROR_NO_TABLE", rp, st);
  if (rc != CM_OK) return rc;
  if (n_points) CM_CUDA(h, cudaMemsetAsync(h->zw.mask.get(), 0, (size_t)n_points * sizeof(unsigned short), st));
  CM_CUDA(h, launch_radius_count(vp, rp, st));
  ++w.launches;
  CM_CUDA(h, cudaEventRecord(w.ev[EV_CENT].get(), st));
  rc = zone_run(h, pts, n_points, st, true, n_clouds);
  if (rc != CM_OK) return rc;
  // the count kernel's verdict on the 2^14-cell bound rides along with the zone sizes: cm_get_zone_out reports it
  CM_CUDA(h, cudaMemcpyAsync(h->zw.report.get() + CM_MAX_ZONES + 2, &vp.ctrl->error, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  h->zw.ror_run = true;
  return CM_OK;
}
}  // namespace

int cm_dev_radius_outlier(cm_handle_t h, const float* xyzi_dev, int64_t n_points, double radius, int min_neighbors,
                          int negative, void* stream) {
  const int64_t begin[2] = {0, n_points};
  return cm_dev_radius_outlier_multi(h, xyzi_dev, begin, 1, radius, min_neighbors, negative, stream);
}

int cm_dev_radius_outlier_multi(cm_handle_t h, const float* xyzi_dev, const int64_t* begin, int n_clouds, double radius,
                                int min_neighbors, int negative, void* stream) {
  if (!h || !begin) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  return radius_outlier_run(h, reinterpret_cast<const float4*>(xyzi_dev), begin, n_clouds, radius, min_neighbors, negative,
                            static_cast<cudaStream_t>(stream));
}

int cm_radius_outlier_multi(cm_handle_t h, const float* xyzi_host, const int64_t* begin, int n_clouds, double radius,
                            int min_neighbors, int negative, float* out_xyzi, uint32_t* out_idx, int64_t capacity,
                            int64_t* out_begin) {
  if (!h || !begin || !out_begin) return CM_E_INVALID;
  if (n_clouds < 1 || n_clouds > CM_MAX_ZONES) return fail(h, CM_E_INVALID, "1 .. %d clouds per call", CM_MAX_ZONES);
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  const float4* pts = nullptr;
  int rc = stage_host_cloud(h, xyzi_host, begin[n_clouds], &pts);
  if (rc == CM_OK) rc = radius_outlier_run(h, pts, begin, n_clouds, radius, min_neighbors, negative, nullptr);
  return rc == CM_OK ? zone_copy_out(h, n_clouds + 1, out_xyzi, out_idx, capacity, out_begin) : rc;
}

int cm_radius_outlier(cm_handle_t h, const float* xyzi_host, int64_t n_points, double radius, int min_neighbors,
                      int negative, float* out_xyzi, uint32_t* out_idx, int64_t capacity, int64_t* n_out) {
  if (!h || !n_out || n_points < 0) return CM_E_INVALID;
  const int64_t begin[2] = {0, n_points};
  int64_t ob[2] = {0, 0};
  const int rc = cm_radius_outlier_multi(h, xyzi_host, begin, 1, radius, min_neighbors, negative, out_xyzi, out_idx, capacity, ob);
  *n_out = ob[1];
  return rc;
}

// ---- statistical outlier removal ----------------------------------------------------------------------------------------
namespace {
int sor_ws_ensure(cm_handle_t h, size_t points) {
  cm_handle_s::SorWs& s = h->sw;
  if (s.cap >= std::max<size_t>(points, 1) && s.stats) return CM_OK;
  const size_t want = std::max<size_t>(points, 1);
  s.sorted_pts.reset(); s.dist.reset(); s.cap = 0;  // the old buffers go before the larger ones are allocated
  CM_CUDA(h, dev_alloc(s.sorted_pts, want));
  CM_CUDA(h, dev_alloc(s.dist, want));
  if (!s.stats) {
    CM_CUDA(h, dev_alloc(s.stats, (size_t)CM_MAX_ZONES));
    CM_CUDA(h, pinned_alloc(s.stats_host, sizeof(SorStats) * CM_MAX_ZONES, cudaHostAllocDefault));
    for (auto& e : s.ev) CM_CUDA(h, create(e, cudaEventCreateWithFlags, cudaEventDefault));
  }
  s.cap = want;
  return CM_OK;
}

// The cell edge of a statistical outlier removal. The result does not depend on it -- the search grows until its bound
// holds -- but the cost does: cells about as wide as the radius that holds mean_k + 1 neighbours of an average point of
// the largest cloud, its points taken as spread over the two largest extents of its bounding box (a LiDAR cloud is a
// surface), so that most searches end after the cube of half-width 1. Never below what keeps every cloud inside the key
// range: at most 2^19 cells across an axis and |x| / edge <= 2^20, which also keeps the float rounding of x * inv below
// 1/8 cell. CM_SOR_CELL=<metres> overrides the estimate (not the key-range floor): tests force tiny and huge cells with it.
double sor_cell_edge(const float (*mn)[3], const float (*mx)[3], const int64_t* n_fin, int n_clouds, int mean_k) {
  double floor_edge = 0.0, edge = 1.0;
  int64_t biggest = 0;
  for (int c = 0; c < n_clouds; ++c) {
    if (n_fin[c] <= 0) continue;
    double e[3];
    for (int a = 0; a < 3; ++a) {
      e[a] = (double)mx[c][a] - (double)mn[c][a];
      const double mag = std::max(std::fabs((double)mn[c][a]), std::fabs((double)mx[c][a]));
      floor_edge = std::max(floor_edge, std::max(mag / 1048576.0, e[a] / 524288.0));
    }
    std::sort(e, e + 3, [](double x, double y) { return x > y; });
    double ec = 1.0;
    if (e[1] > 0.0) ec = std::sqrt((mean_k + 1.0) * e[0] * e[1] / (3.141592653589793 * (double)n_fin[c]));
    else if (e[0] > 0.0) ec = (mean_k + 1.0) * e[0] / (2.0 * (double)n_fin[c]);
    if (n_fin[c] > biggest) { biggest = n_fin[c]; edge = ec; }
  }
  const char* forced = getenv("CM_SOR_CELL");
  if (forced && atof(forced) > 0.0) edge = atof(forced);
  edge = std::max(edge, floor_edge * (1.0 + 1.0 / 1024.0));
  return std::min(std::max(edge, 1e-30), 1e36);  // 1 / edge stays a normal float
}

// output zone k = the survivors of cloud k
int statistical_outlier_run(cm_handle_t h, const float4* pts, const int64_t* begin, int n_clouds, const cm_sor_cfg_t* cfg,
                            cudaStream_t st) {
  if (!cfg) return fail(h, CM_E_INVALID, "cfg is NULL");
  if (cfg->mean_k < 1 || cfg->mean_k > CM_SOR_MAX_K) return fail(h, CM_E_INVALID, "mean_k must be 1 .. %d", CM_SOR_MAX_K);
  if (std::isnan(cfg->std_mul)) return fail(h, CM_E_INVALID, "std_mul is NaN");
  if (cfg->sqrt_mode != CM_SOR_SQRT_FLOAT && cfg->sqrt_mode != CM_SOR_SQRT_DOUBLE) return fail(h, CM_E_INVALID, "bad sqrt_mode");
  int rc = check_clouds(h, pts, begin, n_clouds, CM_MAX_ZONES);
  if (rc != CM_OK) return rc;
  const int64_t n_points = begin[n_clouds];
  VoxelParams vp;
  rc = cell_keys_begin(h, pts, begin, n_clouds, vp, st);
  if (rc != CM_OK) return rc;
  rc = sor_ws_ensure(h, (size_t)n_points);
  if (rc != CM_OK) return rc;
  Workspace& w = h->batch;
  cm_handle_s::SorWs& s = h->sw;
  s.ran = false;
  // one round trip: the bounds choose the cell edge, the finite counts are PCL's valid_distances
  FrameAcc acc[CM_MAX_ZONES];
  CM_CUDA(h, cudaMemcpyAsync(acc, vp.acc, sizeof(FrameAcc) * (size_t)n_clouds, cudaMemcpyDeviceToHost, st));
  CM_CUDA(h, cudaStreamSynchronize(st));
  float mn[CM_MAX_ZONES][3], mx[CM_MAX_ZONES][3];
  int64_t n_fin[CM_MAX_ZONES];
  uint32_t too_few = 0;
  for (int c = 0; c < n_clouds; ++c) {
    const int64_t n_here = begin[c + 1] - begin[c];
    n_fin[c] = n_here ? n_here - (int64_t)acc[c].n_invalid : 0;
    for (int a = 0; a < 3; ++a) {
      const uint32_t lo = f32_order_dec(~acc[c].nmin_enc[a]), hi = f32_order_dec(acc[c].max_enc[a]);
      memcpy(&mn[c][a], &lo, 4);
      memcpy(&mx[c][a], &hi, 4);
    }
    s.n_valid[c] = (uint32_t)n_fin[c];
    if (n_fin[c] > 0 && n_fin[c] <= cfg->mean_k) too_few |= 1u << c;
  }
  const float inv = (float)(1.0 / sor_cell_edge(mn, mx, n_fin, n_clouds, cfg->mean_k));
  rc = cell_keys_sort(h, vp, inv, st);
  if (rc != CM_OK) return rc;
  SorParams sp;
  sp.mean_k = (uint32_t)cfg->mean_k;
  sp.sqrt_mode = (uint32_t)cfg->sqrt_mode;
  sp.too_few = too_few;
  sp.sorted_pts = s.sorted_pts.get();
  sp.dist = s.dist.get();
  sp.cell = 1.0 / (double)inv;
  RorParams rp{};
  rc = enqueue_cell_table(h, vp, "CM_SOR_NO_TABLE", rp, st);
  if (rc != CM_OK) return rc;
  sp.cell_start = rp.cell_start;
  if (n_points) CM_CUDA(h, cudaMemsetAsync(s.dist.get(), 0, (size_t)n_points * sizeof(float), st));
  s.profiled = h->profiling;
  if (s.profiled) CM_CUDA(h, cudaEventRecord(s.ev[0].get(), st));
  CM_CUDA(h, launch_sor_knn(vp, sp, s.sorted_pts.get(), st));
  w.launches += 2;
  if (s.profiled) CM_CUDA(h, cudaEventRecord(s.ev[1].get(), st));
  SorSumParams q{};
  q.dist = s.dist.get();
  q.n_clouds = (uint32_t)n_clouds;
  for (int c = 0; c <= n_clouds; ++c) q.begin[c] = (uint32_t)begin[c];
  for (int c = 0; c < n_clouds; ++c) q.n_valid[c] = s.n_valid[c];
  q.too_few = too_few;
  q.force_serial = getenv("CM_SOR_SERIAL_SUMS") ? 1u : 0u;  // test hook: the serial chain for every cloud
  q.negative = cfg->negative ? 1u : 0u;
  q.std_mul = cfg->std_mul;
  q.stats = s.stats.get();
  q.mask = h->zw.mask.get();
  CM_CUDA(h, launch_sor_sums(q, st));
  if (s.profiled) CM_CUDA(h, cudaEventRecord(s.ev[2].get(), st));
  CM_CUDA(h, launch_sor_select(q, (uint32_t)n_points, st));
  w.launches += 2;
  CM_CUDA(h, cudaMemcpyAsync(s.stats_host.get(), s.stats.get(), sizeof(SorStats) * (size_t)n_clouds, cudaMemcpyDeviceToHost, st));
  CM_CUDA(h, cudaEventRecord(w.ev[EV_CENT].get(), st));
  rc = zone_run(h, pts, n_points, st, true, n_clouds);
  if (rc != CM_OK) return rc;
  s.stream = st; s.n_clouds = n_clouds; s.n_points = n_points; s.too_few = too_few; s.ran = true;
  return CM_OK;
}
}  // namespace

int cm_dev_statistical_outlier(cm_handle_t h, const float* xyzi_dev, int64_t n_points, const cm_sor_cfg_t* cfg, void* stream) {
  const int64_t begin[2] = {0, n_points};
  return cm_dev_statistical_outlier_multi(h, xyzi_dev, begin, 1, cfg, stream);
}

int cm_dev_statistical_outlier_multi(cm_handle_t h, const float* xyzi_dev, const int64_t* begin, int n_clouds,
                                     const cm_sor_cfg_t* cfg, void* stream) {
  if (!h || !begin) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  return statistical_outlier_run(h, reinterpret_cast<const float4*>(xyzi_dev), begin, n_clouds, cfg,
                                 static_cast<cudaStream_t>(stream));
}

int cm_statistical_outlier_multi(cm_handle_t h, const float* xyzi_host, const int64_t* begin, int n_clouds,
                                 const cm_sor_cfg_t* cfg, float* out_xyzi, uint32_t* out_idx, int64_t capacity,
                                 int64_t* out_begin) {
  if (!h || !begin || !out_begin) return CM_E_INVALID;
  if (n_clouds < 1 || n_clouds > CM_MAX_ZONES) return fail(h, CM_E_INVALID, "1 .. %d clouds per call", CM_MAX_ZONES);
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  const float4* pts = nullptr;
  int rc = stage_host_cloud(h, xyzi_host, begin[n_clouds], &pts);
  if (rc == CM_OK) rc = statistical_outlier_run(h, pts, begin, n_clouds, cfg, nullptr);
  return rc == CM_OK ? zone_copy_out(h, n_clouds + 1, out_xyzi, out_idx, capacity, out_begin) : rc;
}

int cm_statistical_outlier(cm_handle_t h, const float* xyzi_host, int64_t n_points, const cm_sor_cfg_t* cfg,
                           float* out_xyzi, uint32_t* out_idx, int64_t capacity, int64_t* n_out) {
  if (!h || !n_out || n_points < 0) return CM_E_INVALID;
  const int64_t begin[2] = {0, n_points};
  int64_t ob[2] = {0, 0};
  const int rc = cm_statistical_outlier_multi(h, xyzi_host, begin, 1, cfg, out_xyzi, out_idx, capacity, ob);
  *n_out = ob[1];
  return rc;
}

int cm_get_statistical_out(cm_handle_t h, cm_sor_out_t* out) {
  if (!h || !out) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  cm_handle_s::SorWs& s = h->sw;
  if (!s.ran) return fail(h, CM_E_INVALID, "no statistical outlier removal has run on this handle");
  CM_CUDA(h, cudaSetDevice(h->device));
  CM_CUDA(h, cudaStreamSynchronize(s.stream));
  memset(out, 0, sizeof(*out));
  out->distances = s.dist.get();
  out->n_points = s.n_points;
  out->n_clouds = s.n_clouds;
  out->knn_ms = out->sums_ms = -1.f;
  if (s.profiled) {
    if (cudaEventElapsedTime(&out->knn_ms, s.ev[0].get(), s.ev[1].get()) != cudaSuccess) { out->knn_ms = -1.f; cudaGetLastError(); }
    if (cudaEventElapsedTime(&out->sums_ms, s.ev[1].get(), s.ev[2].get()) != cudaSuccess) { out->sums_ms = -1.f; cudaGetLastError(); }
  }
  for (int c = 0; c < s.n_clouds; ++c) {
    const SorStats& st = s.stats_host.get()[c];
    cm_sor_stats_t& o = out->cloud[c];
    o.mean = st.mean; o.stddev = st.stddev; o.threshold = st.threshold;
    o.n_valid = s.n_valid[c];
    o.too_few = (s.too_few >> c) & 1u;
    o.sum_path = (int32_t)st.path;
  }
  return CM_OK;
}

// ---- RANSAC ground plane --------------------------------------------------------------------------------------------------
namespace {
constexpr size_t PLANE_FIRST_BATCH = 32;   // PCL's stopping rule usually ends within ~10 iterations on a ground zone;
constexpr size_t PLANE_SECOND_BATCH = 256;  // the host draws (and the GPU scores) no further ahead than this
constexpr size_t PLANE_BATCH = 1024;  // draws per cloud and batch

int plane_ws_ensure(cm_handle_t h) {
  cm_handle_s::PlaneWs& q = h->pw;
  if (q.cap_draws) return CM_OK;
  q = cm_handle_s::PlaneWs();  // frees what an earlier, failed call left behind
  const size_t draws = PLANE_BATCH * CM_MAX_PLANE_CLOUDS;
  CM_CUDA(h, dev_alloc(q.samples_dev, draws * 3));
  CM_CUDA(h, dev_alloc(q.counts_dev, draws * 2));
  CM_CUDA(h, dev_alloc(q.models_dev, draws));
  CM_CUDA(h, dev_alloc(q.acc_dev, (size_t)16 * CM_MAX_PLANE_CLOUDS));
  CM_CUDA(h, pinned_alloc(q.samples_pin, draws * 3 * sizeof(int32_t), cudaHostAllocDefault));
  CM_CUDA(h, pinned_alloc(q.counts_pin, draws * 2 * sizeof(int32_t), cudaHostAllocDefault));
  CM_CUDA(h, pinned_alloc(q.models_pin, draws * sizeof(float4), cudaHostAllocDefault));
  CM_CUDA(h, pinned_alloc(q.acc_pin, 16 * CM_MAX_PLANE_CLOUDS * sizeof(float), cudaHostAllocDefault));
  q.cap_draws = draws;
  return CM_OK;
}

// SampleConsensusModel::shuffled_indices_ without the O(n) array: only the entries a swap has touched are stored, in a
// small open-addressing table (three swaps per draw; identity everywhere else)
struct ShuffledIndices {
  std::vector<uint32_t> key;  // position + 1 (0 = empty)
  std::vector<int32_t> val;
  size_t used = 0, mask = 0;
  ShuffledIndices() { rehash(256); }
  void rehash(size_t cap) {
    std::vector<uint32_t> ok; std::vector<int32_t> ov;
    ok.swap(key); ov.swap(val);
    key.assign(cap, 0u); val.assign(cap, 0);
    mask = cap - 1; used = 0;
    for (size_t i = 0; i < ok.size(); ++i) if (ok[i]) *slot(ok[i] - 1) = ov[i];
  }
  // the value cell of position `pos`, created with the identity value if absent
  int32_t* slot(uint32_t pos) {
    size_t i = ((size_t)pos * 0x9E3779B1u) & mask;
    while (key[i] && key[i] != pos + 1) i = (i + 1) & mask;
    if (!key[i]) { key[i] = pos + 1; val[i] = (int32_t)pos; ++used; }
    return &val[i];
  }
  int32_t get(int64_t pos) const {
    size_t i = ((size_t)(uint32_t)pos * 0x9E3779B1u) & mask;
    while (key[i] && key[i] != (uint32_t)pos + 1) i = (i + 1) & mask;
    return key[i] ? val[i] : (int32_t)pos;
  }
  void swap(int64_t a, int64_t b) {
    if (a == b) return;
    if ((used + 2) * 2 > mask + 1) rehash((mask + 1) * 2);
    int32_t* pa = slot((uint32_t)a);
    int32_t* pb = slot((uint32_t)b);
    std::swap(*pa, *pb);
  }
};

// Eigen's 4-wide float reduction in the order of the build PCL came from (cm_plane_cfg_t::sum_order)
float sum4_host(float l0, float l1, float l2, float l3, int order) {
  if (order == CM_SUM4_SSE2) return (l0 + l2) + (l1 + l3);
  if (order == CM_SUM4_SSE3) return (l0 + l1) + (l2 + l3);
  return ((l0 + l1) + l2) + l3;
}

// pcl::computeRoots2 (common/impl/eigen.hpp): roots of x^2 - b x + c, with the zero root in front
void plane_roots2(float b, float c, float* roots) {
  roots[0] = 0.0f;
  float d = (float)(b * b - 4.0 * c);
  if (d < 0.0) d = 0.0f;
  const float sd = std::sqrt(d);
  roots[2] = 0.5f * (b + sd);
  roots[1] = 0.5f * (b - sd);
}

// pcl::computeRoots for a symmetric 3x3 float matrix given as xx xy xz yy yz zz; ascending roots
void plane_roots3(const float* a, float* roots) {
  const float xx = a[0], xy = a[1], xz = a[2], yy = a[3], yz = a[4], zz = a[5];
  const float c0 = xx * yy * zz + 2.0f * xy * xz * yz - xx * yz * yz - yy * xz * xz - zz * xy * xy;
  const float c1 = xx * yy - xy * xy + xx * zz - xz * xz + yy * zz - yz * yz;
  const float c2 = xx + yy + zz;
  if (std::fabs(c0) < std::numeric_limits<float>::epsilon()) return plane_roots2(c2, c1, roots);
  const float inv3 = (float)(1.0 / 3.0), sqrt3 = std::sqrt(3.0f);
  const float c2_3 = c2 * inv3;
  float a_3 = (c1 - c2 * c2_3) * inv3;
  if (a_3 > 0.0f) a_3 = 0.0f;
  const float half_b = 0.5f * (c0 + c2_3 * (2.0f * c2_3 * c2_3 - c1));
  float q = half_b * half_b + a_3 * a_3 * a_3;
  if (q > 0.0f) q = 0.0f;
  const float rho = std::sqrt(-a_3);
  const float theta = std::atan2(std::sqrt(-q), half_b) * inv3;
  const float ct = std::cos(theta), sn = std::sin(theta);
  roots[0] = c2_3 + 2.0f * rho * ct;
  roots[1] = c2_3 - rho * (ct + sqrt3 * sn);
  roots[2] = c2_3 - rho * (ct - sqrt3 * sn);
  if (roots[0] >= roots[1]) std::swap(roots[0], roots[1]);
  if (roots[1] >= roots[2]) {
    std::swap(roots[1], roots[2]);
    if (roots[0] >= roots[1]) std::swap(roots[0], roots[1]);
  }
  if (roots[0] <= 0.0f) plane_roots2(c2, c1, roots);
}

// SampleConsensusModelPlane::optimizeModelCoefficients after the running sums: mean, covariance, pcl::eigen33's
// eigenvector of the smallest eigenvalue, d = -n . centroid. sums = xx xy xz yy yz zz x y z (PCL-order float sums).
void plane_refit(const float* sums, uint32_t count, int order, float* coeff) {
  float m[9];
  const float cnt = (float)count;
  for (int i = 0; i < 9; ++i) m[i] = sums[i] / cnt;
  float cov[6] = {m[0] - m[6] * m[6], m[1] - m[6] * m[7], m[2] - m[6] * m[8],
                  m[3] - m[7] * m[7], m[4] - m[7] * m[8], m[5] - m[8] * m[8]};
  float scale = 0.0f;
  for (int i = 0; i < 6; ++i) scale = std::max(scale, std::fabs(cov[i]));
  if (scale <= std::numeric_limits<float>::min()) scale = 1.0f;
  for (int i = 0; i < 6; ++i) cov[i] = cov[i] / scale;
  float roots[3];
  plane_roots3(cov, roots);
  const float r0[3] = {cov[0] - roots[0], cov[1], cov[2]};
  const float r1[3] = {cov[1], cov[3] - roots[0], cov[4]};
  const float r2[3] = {cov[2], cov[4], cov[5] - roots[0]};
  auto cross = [](const float* u, const float* v, float* o) {
    o[0] = u[1] * v[2] - u[2] * v[1];
    o[1] = u[2] * v[0] - u[0] * v[2];
    o[2] = u[0] * v[1] - u[1] * v[0];
  };
  float v01[3], v02[3], v12[3];
  cross(r0, r1, v01); cross(r0, r2, v02); cross(r1, r2, v12);
  auto len2 = [](const float* u) { return u[0] * u[0] + u[1] * u[1] + u[2] * u[2]; };
  const float l01 = len2(v01), l02 = len2(v02), l12 = len2(v12);
  const float* pick; float len;
  if (l01 >= l02 && l01 >= l12) { pick = v01; len = l01; }
  else if (l02 >= l01 && l02 >= l12) { pick = v02; len = l02; }
  else { pick = v12; len = l12; }
  const float nrm = std::sqrt(len);
  for (int i = 0; i < 3; ++i) coeff[i] = pick[i] / nrm;
  coeff[3] = -1.0f * sum4_host(coeff[0] * m[6], coeff[1] * m[7], coeff[2] * m[8], 0.0f * 1.0f, order);
}

// RandomSampleConsensus::computeModel of one cloud, fed batch by batch
struct PlaneSearch {
  uint32_t n = 0;
  std::mt19937 engine;
  ShuffledIndices shuffled;
  int iterations = 0, draws = 0, bad_run = 0;
  long long best = -(long long)std::numeric_limits<int>::max();
  double k = 1.0, one_over_indices = 0.0;
  bool stop = false, found = false;
  bool running() const { return n >= 3 && !stop && iterations < k; }
};

// clouds = the ranges [begin[k], begin[k+1]) of pts; out[n_clouds]; output zones 2k = inliers, 2k + 1 = rest of cloud k
int plane_ransac_run(cm_handle_t h, const float4* pts, const int64_t* begin, int n_clouds, const cm_plane_cfg_t& cfg,
                     cm_plane_t* out, cudaStream_t st) {
  int rc = check_clouds(h, pts, begin, n_clouds, CM_MAX_PLANE_CLOUDS);
  if (rc != CM_OK) return rc;
  const int64_t n_points = begin[n_clouds];
  if (n_points > 0x7FFFFFF0ll) return fail(h, CM_E_INVALID, "bad n_points");
  if (cfg.max_iterations < 0 || cfg.sum_order < 0 || cfg.sum_order > 2) return fail(h, CM_E_INVALID, "bad plane settings");
  rc = zone_ws_ensure(h, (size_t)n_points);
  if (rc != CM_OK) return rc;
  rc = plane_ws_ensure(h);
  if (rc != CM_OK) return rc;
  cm_handle_s::PlaneWs& q = h->pw;
  // PCL compares the float distance with the double threshold: the smallest float >= threshold decides the same way
  float thr = (float)cfg.distance_threshold;
  if ((double)thr < cfg.distance_threshold) thr = std::nextafter(thr, std::numeric_limits<float>::infinity());
  int64_t launches = 0;

  PlaneParams pp{};
  pp.pts = pts; pp.n_clouds = (uint32_t)n_clouds; pp.draw_stride = (uint32_t)PLANE_BATCH;
  pp.threshold = thr; pp.sum_order = (uint32_t)cfg.sum_order;
  pp.samples = q.samples_dev.get(); pp.models = q.models_dev.get(); pp.counts = q.counts_dev.get(); pp.good = q.counts_dev.get() + q.cap_draws;
  std::vector<PlaneSearch> search((size_t)n_clouds);
  // CM_PLANE_TRACE=1: where the wall time of a call goes (host draws / scoring round trips / select + refit), to stderr
  static const bool trace = getenv("CM_PLANE_TRACE") != nullptr;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration<double, std::micro>(b - a).count();
  };
  double t_draw = 0, t_score = 0, t_walk = 0;
  int rounds = 0;
  const auto t_begin = now();
  for (int c = 0; c <= n_clouds; ++c) pp.begin[c] = (uint32_t)begin[c];
  for (int c = 0; c < n_clouds; ++c) {
    PlaneSearch& s = search[(size_t)c];
    s.n = (uint32_t)(begin[c + 1] - begin[c]);
    s.engine.seed(cfg.seed);
    s.one_over_indices = s.n ? 1.0 / (double)s.n : 0.0;
    memset(&out[c], 0, sizeof(out[c]));
    out[c].sample[0] = out[c].sample[1] = out[c].sample[2] = -1;
  }
  const double log_probability = std::log(1.0 - cfg.probability);

  // the draw streams of SampleConsensusModel::getSamples, scored a batch at a time
  size_t batch = PLANE_FIRST_BATCH;
  for (;;) {
    bool any = false;
    const auto t0 = now();
    for (int c = 0; c < n_clouds; ++c) {
      PlaneSearch& s = search[(size_t)c];
      pp.n_draws[c] = 0;
      if (!s.running()) continue;
      any = true;
      pp.n_draws[c] = (uint32_t)batch;
      int32_t* smp = q.samples_pin.get() + 3 * (size_t)c * PLANE_BATCH;
      for (size_t d = 0; d < batch; ++d) {
        for (int64_t i = 0; i < 3; ++i) {
          const uint64_t r = (uint64_t)((uint32_t)s.engine() >> 1);  // boost::uniform_int<>(0, INT_MAX) on mt19937
          s.shuffled.swap(i, i + (int64_t)(r % (uint64_t)(s.n - i)));
        }
        for (int64_t i = 0; i < 3; ++i) smp[3 * d + i] = s.shuffled.get(i);
      }
    }
    if (!any) break;
    const auto t1 = now();
    const size_t used = (size_t)(n_clouds - 1) * PLANE_BATCH + batch;  // the per-draw arrays up to the last cloud's batch
    CM_CUDA(h, cudaMemcpyAsync(q.samples_dev.get(), q.samples_pin.get(), used * 3 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CM_CUDA(h, cudaMemsetAsync(q.counts_dev.get(), 0, used * sizeof(int32_t), st));
    CM_CUDA(h, launch_plane_score(pp, st));
    ++launches;
    CM_CUDA(h, cudaMemcpyAsync(q.counts_pin.get(), q.counts_dev.get(), used * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CM_CUDA(h, cudaMemcpyAsync(q.counts_pin.get() + q.cap_draws, q.counts_dev.get() + q.cap_draws, used * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CM_CUDA(h, cudaMemcpyAsync(q.models_pin.get(), q.models_dev.get(), used * sizeof(float4), cudaMemcpyDeviceToHost, st));
    CM_CUDA(h, cudaStreamSynchronize(st));
    const auto t2 = now();
    for (int c = 0; c < n_clouds; ++c) {
      PlaneSearch& s = search[(size_t)c];
      const size_t n_draws = pp.n_draws[c], off = (size_t)c * PLANE_BATCH;
      const int32_t* counts = q.counts_pin.get() + off;
      const int32_t* good = q.counts_pin.get() + q.cap_draws + off;
      for (size_t d = 0; d < n_draws && s.running(); ++d) {
        ++s.draws;
        if (!good[d]) {  // getSamples draws again; after max_sample_checks_ (1000) failures in a row it gives up
          if (++s.bad_run == 1000) s.stop = true;
          continue;
        }
        s.bad_run = 0;
        if ((long long)counts[d] > s.best) {
          s.best = counts[d];
          s.found = true;
          out[c].best_count = counts[d];
          for (int i = 0; i < 3; ++i) out[c].sample[i] = q.samples_pin.get()[3 * (off + d) + i];
          const float4 m = q.models_pin.get()[off + d];
          out[c].coeff_ransac[0] = m.x; out[c].coeff_ransac[1] = m.y; out[c].coeff_ransac[2] = m.z; out[c].coeff_ransac[3] = m.w;
          const double w = (double)s.best * s.one_over_indices;
          double p_no_outliers = 1.0 - std::pow(w, 3.0);
          p_no_outliers = std::max(std::numeric_limits<double>::epsilon(), p_no_outliers);
          p_no_outliers = std::min(1.0 - std::numeric_limits<double>::epsilon(), p_no_outliers);
          s.k = log_probability / std::log(p_no_outliers);
        }
        ++s.iterations;
        if (s.iterations > cfg.max_iterations) s.stop = true;
      }
    }
    batch = batch == PLANE_FIRST_BATCH ? PLANE_SECOND_BATCH : PLANE_BATCH;
    t_draw += us(t0, t1); t_score += us(t1, t2); t_walk += us(t2, now());
    ++rounds;
  }
  const auto t_search = now();

  // what follows the search: zone 2k = inliers of cloud k, zone 2k + 1 = its other points
  PlaneSelect ps{};
  ps.pts = pts; ps.n_clouds = (uint32_t)n_clouds; ps.threshold = thr; ps.mask = h->zw.mask.get();
  for (int c = 0; c <= n_clouds; ++c) ps.begin[c] = (uint32_t)begin[c];
  bool any_found = false;
  for (int c = 0; c < n_clouds; ++c) {
    const PlaneSearch& s = search[(size_t)c];
    out[c].found = s.found ? 1 : 0;
    out[c].iterations = s.iterations;
    out[c].draws = s.draws;
    memcpy(out[c].coeff, out[c].coeff_ransac, sizeof(out[c].coeff));
    ps.found[c] = s.found ? 1u : 0u;
    ps.coeff[c] = make_float4(out[c].coeff[0], out[c].coeff[1], out[c].coeff[2], out[c].coeff[3]);
    any_found = any_found || s.found;
  }
  if (any_found && cfg.optimize) {
    // optimizeModelCoefficients on the inliers of the RANSAC model: the running sums on the device, the 3 x 3 part here
    CM_CUDA(h, launch_plane_moments(ps, (uint32_t)cfg.sum_order, q.acc_dev.get(), st));
    ++launches;
    CM_CUDA(h, cudaMemcpyAsync(q.acc_pin.get(), q.acc_dev.get(), (size_t)16 * n_clouds * sizeof(float), cudaMemcpyDeviceToHost, st));
    CM_CUDA(h, cudaStreamSynchronize(st));
    for (int c = 0; c < n_clouds; ++c) {
      uint32_t n_in;
      memcpy(&n_in, q.acc_pin.get() + 16 * c + 9, sizeof(n_in));
#ifdef CM_PLANE_CYCLES
      if (trace) {
        uint32_t cyc[2];
        memcpy(cyc, q.acc_pin.get() + 16 * c + 10, sizeof(cyc));
        fprintf(stderr, "[cm plane] cloud %d: moments kernel %u cycles, adding warp busy %u cycles, %u inliers\n", c, cyc[0], cyc[1], n_in);
      }
#endif
      if (!search[(size_t)c].found || n_in < 4) continue;  // below 4 inliers PCL keeps the RANSAC model
      plane_refit(q.acc_pin.get() + 16 * c, n_in, cfg.sum_order, out[c].coeff);
      ps.coeff[c] = make_float4(out[c].coeff[0], out[c].coeff[1], out[c].coeff[2], out[c].coeff[3]);
    }
  }
  // selectWithinDistance with the final model + the two ExtractIndices passes
  CM_CUDA(h, launch_plane_select(ps, (uint32_t)cfg.sum_order, st));
  ++launches;
  rc = zone_run(h, pts, n_points, st, true, 2 * n_clouds);
  if (rc != CM_OK) return rc;
  launches += h->zw.launches;
  cm_zone_out_t zo;
  rc = zone_out_locked(h, &zo);
  if (rc != CM_OK) return rc;
  h->zw.launches = launches;
  for (int c = 0; c < n_clouds; ++c) out[c].n_inliers = zo.begin[2 * c + 1] - zo.begin[2 * c];
  if (trace)
    fprintf(stderr, "[cm plane] clouds %d points %lld: %d scoring rounds (host draws %.1f us, GPU round trips %.1f us, stopping rule %.1f us), "
            "refit + select + compaction %.1f us, total %.1f us, %lld launches\n", n_clouds, (long long)n_points, rounds, t_draw, t_score,
            t_walk, us(t_search, now()), us(t_begin, now()), (long long)launches);
  return CM_OK;
}
}  // namespace

int cm_dev_plane_ransac_multi(cm_handle_t h, const float* xyzi_dev, const int64_t* begin, int n_clouds,
                              const cm_plane_cfg_t* cfg, cm_plane_t* out, void* stream) {
  if (!h || !cfg || !out || !begin) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  return plane_ransac_run(h, reinterpret_cast<const float4*>(xyzi_dev), begin, n_clouds, *cfg, out, static_cast<cudaStream_t>(stream));
}

int cm_dev_plane_ransac(cm_handle_t h, const float* xyzi_dev, int64_t n_points, const cm_plane_cfg_t* cfg, cm_plane_t* out,
                        void* stream) {
  const int64_t begin[2] = {0, n_points};
  return cm_dev_plane_ransac_multi(h, xyzi_dev, begin, 1, cfg, out, stream);
}

int cm_plane_ransac_multi(cm_handle_t h, const float* xyzi_host, const int64_t* begin, int n_clouds, const cm_plane_cfg_t* cfg,
                          cm_plane_t* out, float* out_xyzi, uint32_t* out_idx, int64_t capacity, int64_t* out_begin) {
  if (!h || !cfg || !out || !out_begin || !begin) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  if (n_clouds < 1 || n_clouds > CM_MAX_PLANE_CLOUDS) return fail(h, CM_E_INVALID, "1 .. %d clouds per call", CM_MAX_PLANE_CLOUDS);
  const float4* pts = nullptr;
  int rc = stage_host_cloud(h, xyzi_host, begin[n_clouds], &pts);
  if (rc == CM_OK) rc = plane_ransac_run(h, pts, begin, n_clouds, *cfg, out, nullptr);
  return rc == CM_OK ? zone_copy_out(h, 2 * n_clouds + 1, out_xyzi, out_idx, capacity, out_begin) : rc;
}

int cm_plane_ransac(cm_handle_t h, const float* xyzi_host, int64_t n_points, const cm_plane_cfg_t* cfg, cm_plane_t* out,
                    float* out_xyzi, uint32_t* out_idx, int64_t capacity, int64_t* out_begin) {
  if (n_points < 0) return CM_E_INVALID;
  const int64_t begin[2] = {0, n_points};
  return cm_plane_ransac_multi(h, xyzi_host, begin, 1, cfg, out, out_xyzi, out_idx, capacity, out_begin);
}

// ---- the body of a proceedX in one call ---------------------------------------------------------------------------------------
namespace {
int proceed_ws_ensure(cm_handle_t h, size_t points) {
  cm_handle_s::ProceedWs& w = h->prz;
  const size_t want = std::max<size_t>({points, (size_t)h->cfg.max_batch_points, (size_t)1});
  if (w.cap >= want) return CM_OK;
  w = cm_handle_s::ProceedWs();  // the old buffers go before the larger ones are allocated
  CM_CUDA(h, dev_alloc(w.low, want));
  CM_CUDA(h, dev_alloc(w.high, 2 * want));
  CM_CUDA(h, dev_alloc(w.rest, want));
  CM_CUDA(h, dev_alloc(w.planes, want));
  CM_CUDA(h, dev_alloc(w.no_ground, 2 * want));
  CM_CUDA(h, dev_alloc(w.ground, 2 * want));
  w.cap = want;
  return CM_OK;
}

int proceed_run(cm_handle_t h, const float4* roi, int64_t n, const cm_proceed_cfg_t& cfg, cm_proceed_out_t* out, cudaStream_t st) {
  if (cfg.n_parts < 1 || cfg.n_parts > CM_MAX_PROCEED_PARTS) return fail(h, CM_E_INVALID, "1 .. %d parts", CM_MAX_PROCEED_PARTS);
  if (n < 0 || n > 0x7FFFFFF0ll) return fail(h, CM_E_INVALID, "bad n_points");
  int ground_of[CM_MAX_PROCEED_PARTS], plain_of[CM_MAX_PROCEED_PARTS];
  int G = 0, P = 0;
  for (int k = 0; k < cfg.n_parts; ++k) {
    ground_of[k] = plain_of[k] = -1;
    if (cfg.part[k].ground_removal) ground_of[k] = G++; else plain_of[k] = P++;
  }
  if (2 * G + P > CM_MAX_ZONES || G > CM_MAX_PLANE_CLOUDS) return fail(h, CM_E_INVALID, "too many parts for one pass");
  int rc = ensure_batch_ws(h);
  if (rc != CM_OK) return rc;
  if (G > 0 && (uint32_t)G > h->batch.cap_frames)
    return fail(h, CM_E_CAPACITY, "%d ground-removal parts need max_batch_frames >= %d (handle has %u)", G, G, h->batch.cap_frames);
  rc = proceed_ws_ensure(h, (size_t)n);
  if (rc != CM_OK) return rc;
  cm_handle_s::ProceedWs& w = h->prz;
  memset(out, 0, sizeof(*out));
  out->no_ground_xyzi = reinterpret_cast<const float*>(w.no_ground.get());
  out->ground_xyzi = reinterpret_cast<const float*>(w.ground.get());
  out->n_planes = G;
  // ---- one zone-slicing pass: zones [0, G) the ground windows, [G, 2G) the upper windows, [2G, 2G + P) the plain parts
  const ZoneSet saved = h->zones;
  {
    std::vector<cm_zone_t> zones((size_t)(2 * G + P));
    for (int k = 0; k < cfg.n_parts; ++k) {
      const cm_proceed_part_t& pt = cfg.part[k];
      const cm_pass_t x = {0, pt.deviation, pt.deviation + pt.length, 0};  // float sum, as getCloudPart passes it to setFilterLimits
      if (ground_of[k] >= 0) {
        cm_zone_t& lo = zones[(size_t)ground_of[k]];
        cm_zone_t& hi = zones[(size_t)(G + ground_of[k])];
        lo.n_pass = 2; lo.pass[0] = x; lo.pass[1] = cm_pass_t{2, -pt.z_max_ground, pt.z_max_ground, 0};
        // `z_max_ground + 0.01` is a double sum narrowed to float by setFilterLimits(const float&, const float&) (:88)
        hi.n_pass = 2; hi.pass[0] = x; hi.pass[1] = cm_pass_t{2, (float)((double)pt.z_max_ground + 0.01), cfg.roi_z_max, 0};
      } else {
        cm_zone_t& pl = zones[(size_t)(2 * G + plain_of[k])];
        pl.n_pass = 1; pl.pass[0] = x;
      }
    }
    rc = make_zone_set(h, 2 * G + P, zones.data(), h->zones);
  }
  if (rc == CM_OK) rc = zone_run(h, roi, n, st);
  h->zones = saved;
  if (rc != CM_OK) return rc;
  cm_zone_out_t zo;
  rc = zone_out_locked(h, &zo);
  ++out->host_syncs;
  if (rc != CM_OK) return rc;
  const int64_t n_low = zo.begin[G], n_high = zo.begin[2 * G + P] - n_low;
  if ((size_t)n_low > w.cap || (size_t)n_high > 2 * w.cap) return fail(h, CM_E_CAPACITY, "zone windows larger than the workspace");
  if (n_low) CM_CUDA(h, cudaMemcpyAsync(w.low.get(), zo.xyzi, (size_t)n_low * 16, cudaMemcpyDeviceToDevice, st));
  if (n_high) CM_CUDA(h, cudaMemcpyAsync(w.high.get(), zo.xyzi + n_low * 4, (size_t)n_high * 16, cudaMemcpyDeviceToDevice, st));
  int64_t zb[CM_MAX_ZONES + 1];
  for (int z = 0; z <= 2 * G + P; ++z) zb[z] = zo.begin[z];

  // ---- one multi-cloud plane search over the ground windows, one multi-cloud outlier removal over what is not ground
  int64_t pb[2 * CM_MAX_PLANE_CLOUDS + 1] = {0}, kb[CM_MAX_PLANE_CLOUDS + 1] = {0}, rb[CM_MAX_PLANE_CLOUDS + 1] = {0};
  const float4* kept = nullptr;
  if (G > 0) {
    rc = plane_ransac_run(h, w.low.get(), zb, G, cfg.plane, out->plane, st);  // ends with the sizes on the host
    out->host_syncs += 2 + (cfg.plane.optimize ? 1 : 0);
    if (rc != CM_OK) return rc;
    rc = zone_out_locked(h, &zo);
    if (rc != CM_OK) return rc;
    for (int z = 0; z <= 2 * G; ++z) pb[z] = zo.begin[z];
    if (pb[2 * G]) CM_CUDA(h, cudaMemcpyAsync(w.planes.get(), zo.xyzi, (size_t)pb[2 * G] * 16, cudaMemcpyDeviceToDevice, st));
    for (int c = 0; c < G; ++c) {  // the non-ground points of every window side by side
      const int64_t cnt = pb[2 * c + 2] - pb[2 * c + 1];
      if (cnt) CM_CUDA(h, cudaMemcpyAsync(w.rest.get() + rb[c], w.planes.get() + pb[2 * c + 1], (size_t)cnt * 16, cudaMemcpyDeviceToDevice, st));
      rb[c + 1] = rb[c] + cnt;
    }
    rc = radius_outlier_run(h, w.rest.get(), rb, G, cfg.radius, cfg.min_neighbors, 0, st);
    if (rc != CM_OK) return rc;
    rc = zone_out_locked(h, &zo);
    out->host_syncs += 2;
    if (rc != CM_OK) return rc;
    for (int c = 0; c <= G; ++c) kb[c] = zo.begin[c];
    kept = reinterpret_cast<const float4*>(zo.xyzi);
  }
  // ---- the appends, in part order
  int64_t n_ng = 0, n_g = 0;
  for (int k = 0; k < cfg.n_parts; ++k) {
    if (ground_of[k] >= 0) {
      const int c = ground_of[k];
      int64_t cnt = kb[c + 1] - kb[c];                    // outlierRemoval(no_ground_cloud_ptr) ...
      if (cnt) CM_CUDA(h, cudaMemcpyAsync(w.no_ground.get() + n_ng, kept + kb[c], (size_t)cnt * 16, cudaMemcpyDeviceToDevice, st));
      n_ng += cnt;
      cnt = zb[G + c + 1] - zb[G + c];                    // ... += *no_ground_part_ptr (the upper window)
      if (cnt) CM_CUDA(h, cudaMemcpyAsync(w.no_ground.get() + n_ng, w.high.get() + (zb[G + c] - n_low), (size_t)cnt * 16, cudaMemcpyDeviceToDevice, st));
      n_ng += cnt;
      cnt = pb[2 * c + 1] - pb[2 * c];                    // ground: the inliers
      if (cnt) CM_CUDA(h, cudaMemcpyAsync(w.ground.get() + n_g, w.planes.get() + pb[2 * c], (size_t)cnt * 16, cudaMemcpyDeviceToDevice, st));
      n_g += cnt;
    } else {
      const int z = 2 * G + plain_of[k];
      const int64_t cnt = zb[z + 1] - zb[z];
      if (cnt) CM_CUDA(h, cudaMemcpyAsync(w.no_ground.get() + n_ng, w.high.get() + (zb[z] - n_low), (size_t)cnt * 16, cudaMemcpyDeviceToDevice, st));
      n_ng += cnt;
    }
  }
  out->n_no_ground = n_ng;
  out->n_ground = n_g;
  return CM_OK;
}
}  // namespace

int cm_dev_proceed_zones(cm_handle_t h, const float* roi_xyzi_dev, int64_t n_points, const cm_proceed_cfg_t* cfg,
                         cm_proceed_out_t* out, void* stream) {
  if (!h || !cfg || !out) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  const int rc = check_dev_cloud(h, roi_xyzi_dev, n_points);
  if (rc != CM_OK) return rc;
  return proceed_run(h, reinterpret_cast<const float4*>(roi_xyzi_dev), n_points, *cfg, out, static_cast<cudaStream_t>(stream));
}

int cm_proceed_zones(cm_handle_t h, const float* roi_xyzi_host, int64_t n_points, const cm_proceed_cfg_t* cfg, float* out_no_ground,
                     int64_t no_ground_capacity, int64_t* n_no_ground, float* out_ground, int64_t ground_capacity, int64_t* n_ground,
                     cm_plane_t* out_planes) {
  if (!h || !cfg || !n_no_ground || !n_ground || n_points < 0 || (n_points > 0 && !roi_xyzi_host)) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  const float4* roi = nullptr;
  int rc = stage_host_cloud(h, roi_xyzi_host, n_points, &roi);
  if (rc != CM_OK) return rc;
  cm_proceed_out_t po;
  rc = proceed_run(h, roi, n_points, *cfg, &po, nullptr);
  if (rc != CM_OK) return rc;
  *n_no_ground = po.n_no_ground;
  *n_ground = po.n_ground;
  if (out_planes) for (int c = 0; c < po.n_planes; ++c) out_planes[c] = po.plane[c];
  if (po.n_no_ground > no_ground_capacity || po.n_ground > ground_capacity)
    return fail(h, CM_E_CAPACITY, "%lld / %lld points, caller capacities %lld / %lld", (long long)po.n_no_ground, (long long)po.n_ground,
                (long long)no_ground_capacity, (long long)ground_capacity);
  if (out_no_ground && po.n_no_ground) CM_CUDA(h, cudaMemcpyAsync(out_no_ground, po.no_ground_xyzi, (size_t)po.n_no_ground * 16, cudaMemcpyDeviceToHost, nullptr));
  if (out_ground && po.n_ground) CM_CUDA(h, cudaMemcpyAsync(out_ground, po.ground_xyzi, (size_t)po.n_ground * 16, cudaMemcpyDeviceToHost, nullptr));
  CM_CUDA(h, cudaStreamSynchronize(nullptr));
  return CM_OK;
}

// ---- giant-cloud mode behind one call: C++ + NCCL ----------------------------------------------------------------------------
namespace {
// NCCL entry points resolved at run time: libcloud_merger_gpu.so carries no link-time dependency on libnccl, so a process that
// never uses the giant-cloud mode does not need it, and a process that already holds a libnccl.so.2 (PyTorch ships its own)
// keeps using that one copy.
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string why;
};
NcclApi* nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    api.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);           // the copy the process already has, if any
    if (!api.lib) api.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!api.lib) api.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!api.lib) { api.why = std::string("libnccl.so.2 not found: ") + (dlerror() ? dlerror() : ""); return; }
    bool ok = true;
    auto sym = [&](const char* name) { void* p = dlsym(api.lib, name); if (!p) { ok = false; api.why = std::string("missing NCCL symbol ") + name; } return p; };
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
    api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(sym("ncclAllReduce"));
    api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
    api.Send = reinterpret_cast<decltype(api.Send)>(sym("ncclSend"));
    api.Recv = reinterpret_cast<decltype(api.Recv)>(sym("ncclRecv"));
    api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
    api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
    if (!ok) api.lib = nullptr;
  });
  return api.lib ? &api : nullptr;
}
static_assert(sizeof(ncclUniqueId) == CM_GIANT_ID_BYTES, "ncclUniqueId is 128 bytes");
}  // namespace

struct cm_giant_s {
  cm_handle_t h = nullptr;
  int rank = 0, world = 1;
  ncclComm_t comm = nullptr;
  NcclApi* api = nullptr;
  uint32_t bins = 1u << 14;
  DevPtr<GiantPlan> plan;               // device
  DevPtr<unsigned long long> hist;      // device [bins]
  DevPtr<uint32_t> counts;              // device [world][CM_MAX_ZONES + 2]: every rank's zone_begin
  DevPtr<float4> recv;                  // device [recv_cap]: what the all-to-all delivers
  size_t recv_cap = 0;
  HostPtr<GiantPlan> plan_pin;          // pinned mirrors
  HostPtr<uint32_t> counts_pin;         // [world][stride] + 1: the overflow word of the peer exchange
  // the exchange fused into the grouping kernel: every rank's receive buffer mapped here through CUDA IPC
  bool p2p = false;
  float4* peer_recv[CM_MAX_ZONES] = {};
  DevPtr<uint32_t> p2p_words;           // device: [0..world) remote_base, [world] barrier word, [world + 1] my receive capacity
  Event plan_ready;                     // the host waits for the counts, not for the exchange
  Event prof[5];                        // stage boundaries (cm_set_profiling)
  std::string err;
};

namespace {
int gfail(cm_giant_t g, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g->err = buf;
  if (g->h) g->h->last_error = buf;
  return code;
}
#define CM_G_CUDA(g, expr)                                                                                  \
  do {                                                                                                      \
    cudaError_t e__ = (expr);                                                                               \
    if (e__ != cudaSuccess) return gfail(g, CM_E_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)
#define CM_G_NCCL(g, expr)                                                                                  \
  do {                                                                                                      \
    ncclResult_t r__ = (expr);                                                                              \
    if (r__ != ncclSuccess) return gfail(g, CM_E_CUDA, "%s: NCCL %s (%s:%d)", #expr, (g)->api->GetErrorString(r__), __FILE__, __LINE__); \
  } while (0)
constexpr int kCountStride = CM_MAX_ZONES + 2;

// Maps every peer's receive buffer into this process (CUDA IPC; NVLink peer access is enabled lazily by the open). All or
// nothing: a rank that could not map a peer (two ranks in one process, no P2P between the devices) makes everybody fall back
// to the NCCL exchange, agreed through an all-reduce. Runs on the legacy stream inside cm_giant_create.
void giant_setup_p2p(cm_giant_t g) {
  const char* off = getenv("CM_GIANT_NO_P2P");
  int want = (off && off[0] == '1') ? 0 : 1;
  const int W = g->world;
  cudaIpcMemHandle_t mine;
  memset(&mine, 0, sizeof(mine));
  if (want && cudaIpcGetMemHandle(&mine, g->recv.get()) != cudaSuccess) { want = 0; cudaGetLastError(); }
  DevPtr<cudaIpcMemHandle_t> all_dev;
  DevPtr<int> ok_dev;
  std::vector<cudaIpcMemHandle_t> all((size_t)W);
  int ok = want;
  if (dev_alloc(all_dev, (size_t)W + 1, 0) != cudaSuccess || dev_alloc(ok_dev, 1, 0) != cudaSuccess) { cudaGetLastError(); ok = 0; }
  // every rank takes part in both collectives whatever its own state, or the others would hang
  if (all_dev && ok_dev) {
    cudaMemcpy(all_dev.get() + W, &mine, sizeof(mine), cudaMemcpyHostToDevice);
    if (g->api->AllGather(all_dev.get() + W, all_dev.get(), sizeof(mine), ncclUint8, g->comm, nullptr) != ncclSuccess) ok = 0;
    if (cudaMemcpy(all.data(), all_dev.get(), sizeof(mine) * (size_t)W, cudaMemcpyDeviceToHost) != cudaSuccess) { ok = 0; cudaGetLastError(); }
  }
  int opened = 0;
  if (ok) {
    for (int r = 0; r < W && ok; ++r) {
      if (r == g->rank) { g->peer_recv[r] = g->recv.get(); continue; }
      void* p = nullptr;
      if (cudaIpcOpenMemHandle(&p, all[(size_t)r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; cudaGetLastError(); break; }
      g->peer_recv[r] = static_cast<float4*>(p);
      ++opened;
    }
  }
  if (all_dev && ok_dev) {
    cudaMemcpy(ok_dev.get(), &ok, sizeof(int), cudaMemcpyHostToDevice);
    int agreed = 0;
    if (g->api->AllReduce(ok_dev.get(), ok_dev.get(), 1, ncclInt32, ncclMin, g->comm, nullptr) == ncclSuccess &&
        cudaMemcpy(&agreed, ok_dev.get(), sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess) ok = ok && agreed;
    else ok = 0;
  }
  if (ok && (dev_alloc(g->p2p_words, (size_t)W + 2, 0) != cudaSuccess ||
             create(g->plan_ready, cudaEventCreateWithFlags, cudaEventDisableTiming) != cudaSuccess)) { ok = 0; cudaGetLastError(); }
  if (ok) {
    std::vector<uint32_t> init((size_t)W + 2, 0u);
    init[(size_t)W + 1] = (uint32_t)std::min<size_t>(g->recv_cap, 0xFFFFFFF0u);
    cudaMemcpy(g->p2p_words.get(), init.data(), sizeof(uint32_t) * init.size(), cudaMemcpyHostToDevice);
  }
  if (!ok) {
    for (int r = 0; r < W; ++r) {
      if (r != g->rank && g->peer_recv[r]) cudaIpcCloseMemHandle(g->peer_recv[r]);
      g->peer_recv[r] = nullptr;
    }
    cudaGetLastError();
  }
  (void)opened;
  g->p2p = ok != 0;
}

// The part of cm_giant_create that can fail: the communicator, the batch workspace and the giant-cloud buffers.
int giant_setup(cm_giant_t g, const void* nccl_id) {
  cm_handle_t h = g->h;
  if (g->world > 1 && nccl_id) {
    g->api = nccl_api();
    if (!g->api) { h->last_error = "NCCL unavailable"; return CM_E_CUDA; }
    ncclUniqueId id;
    memcpy(&id, nccl_id, sizeof(id));
    const ncclResult_t r = g->api->CommInitRank(&g->comm, g->world, id, g->rank);
    if (r != ncclSuccess) { h->last_error = std::string("ncclCommInitRank: ") + g->api->GetErrorString(r); return CM_E_CUDA; }
  }
  int rc = ensure_batch_ws(h);
  if (rc != CM_OK) return rc;
  g->recv_cap = h->batch.cap_points;
  if (dev_alloc(g->plan, 1, 0) != cudaSuccess || dev_alloc(g->hist, g->bins, 0) != cudaSuccess ||
      dev_alloc(g->counts, (size_t)kCountStride * g->world, 0) != cudaSuccess ||
      (g->world > 1 && g->comm && dev_alloc(g->recv, g->recv_cap) != cudaSuccess) ||
      pinned_alloc(g->plan_pin, sizeof(GiantPlan), cudaHostAllocDefault) != cudaSuccess ||
      pinned_alloc(g->counts_pin, sizeof(uint32_t) * (kCountStride * g->world + 1), cudaHostAllocDefault) != cudaSuccess) {
    h->last_error = "cm_giant_create: allocation failed";
    cudaGetLastError();
    return CM_E_CUDA;
  }
  if (g->comm && g->recv) giant_setup_p2p(g);
  return CM_OK;
}
}  // namespace

int cm_giant_unique_id(void* id_bytes) {
  if (!id_bytes) return CM_E_INVALID;
  NcclApi* api = nccl_api();
  if (!api) return CM_E_CUDA;
  ncclUniqueId id;
  if (api->GetUniqueId(&id) != ncclSuccess) return CM_E_CUDA;
  memcpy(id_bytes, &id, sizeof(id));
  return CM_OK;
}

const char* cm_giant_last_error(cm_giant_t g) { return g ? g->err.c_str() : "null giant handle"; }

int cm_giant_create(cm_handle_t h, int rank, int world, const void* nccl_id, cm_giant_t* out) {
  if (!h || !out || world < 1 || world > CM_MAX_ZONES || rank < 0 || rank >= world) return CM_E_INVALID;
  *out = nullptr;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  cm_giant_t g = new (std::nothrow) cm_giant_s();
  if (!g) return CM_E_INTERNAL;
  g->h = h; g->rank = rank; g->world = world;
  const int rc = giant_setup(g, nccl_id);
  if (rc != CM_OK) {  // the buffers go with g, the communicator (if one was made) does not
    if (g->comm) g->api->CommDestroy(g->comm);
    delete g;
    return rc;
  }
  *out = g;
  return CM_OK;
}

int cm_giant_destroy(cm_giant_t g) {
  if (!g) return CM_E_INVALID;
  cudaSetDevice(g->h->device);
  cudaDeviceSynchronize();  // past this rank's last barrier: no peer is still storing into g->recv
  for (int r = 0; r < g->world; ++r)
    if (g->p2p && r != g->rank && g->peer_recv[r]) cudaIpcCloseMemHandle(g->peer_recv[r]);
  if (g->comm && g->api) g->api->CommDestroy(g->comm);
  delete g;
  return CM_OK;
}

int cm_giant_voxelgrid(cm_giant_t g, const float* local_xyzi_dev, int64_t n_local, cm_giant_info_t* info, void* stream) {
  if (!g || n_local < 0 || n_local > 0xFFFFFFF0ll) return CM_E_INVALID;
  cm_handle_t h = g->h;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_G_CUDA(g, cudaSetDevice(h->device));
  if (n_local > 0 && (!local_xyzi_dev || (reinterpret_cast<uintptr_t>(local_xyzi_dev) & 15u))) return gfail(g, CM_E_INVALID, "local_xyzi_dev must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float4* pts = reinterpret_cast<const float4*>(local_xyzi_dev);
  const int W = g->world, me = g->rank;
  int rc = ensure_batch_ws(h);
  if (rc != CM_OK) return rc;
  rc = zone_ws_ensure(h, (size_t)n_local);
  if (rc != CM_OK) return rc;
  Workspace& w = h->batch;
  Ctrl* ctrl = reinterpret_cast<Ctrl*>(w.meta.get() + w.ml.off_ctrl);
  FrameAcc* acc = reinterpret_cast<FrameAcc*>(w.meta.get() + w.ml.off_acc);
  uint32_t* fss = reinterpret_cast<uint32_t*>(w.meta.get() + w.ml.off_fstart);
  cm_giant_info_t gi;
  memset(&gi, 0, sizeof(gi));
  gi.points_local = n_local;
  ZoneParams zp;
  const bool prof = h->profiling;
  if (prof)
    for (auto& e : g->prof) if (!e) CM_G_CUDA(g, create(e, cudaEventCreateWithFlags, cudaEventDefault));
  auto mark = [&](int i) { return prof ? cudaEventRecord(g->prof[i].get(), st) : cudaSuccess; };
  CM_G_CUDA(g, mark(0));
  // ---- global bounding box -> grid, on the device
  CM_G_CUDA(g, cudaMemsetAsync(w.meta.get(), 0, w.ml.zero_bytes, st));
  CM_G_CUDA(g, launch_minmax(pts, (uint32_t)n_local, ctrl, acc, fss, st));
  if (g->comm) CM_G_NCCL(g, g->api->AllReduce(acc, acc, 6, ncclUint32, ncclMax, g->comm, st));  // max_enc[3], nmin_enc[3]
  CM_G_CUDA(g, launch_giant_plan(g->plan.get(), acc, h->inv_leaf, g->bins, st));
  // ---- balancing splitters from the all-reduced histogram of the voxel index, on the device
  if (W > 1) {
    CM_G_CUDA(g, cudaMemsetAsync(g->hist.get(), 0, sizeof(unsigned long long) * g->bins, st));
    CM_G_CUDA(g, launch_giant_hist(pts, (uint32_t)n_local, g->plan.get(), g->bins, g->hist.get(), st));
    if (g->comm) CM_G_NCCL(g, g->api->AllReduce(g->hist.get(), g->hist.get(), g->bins, ncclUint64, ncclSum, g->comm, st));
    CM_G_CUDA(g, launch_giant_splitters(g->plan.get(), g->hist.get(), g->bins, (uint32_t)W, st));
    CM_G_CUDA(g, mark(1));
    // ---- group the block by destination (source order kept inside a destination): the send buffer of the all-to-all
    // (the destination masks are derived inside the count sweep from the device-resident plan)
    if (g->p2p) {
      // count + scan only; the scatter below IS the all-to-all (stores into the owners' receive buffers over NVLink)
      if (in_zone_outputs(h, pts, n_local)) return gfail(g, CM_E_INVALID, "the input cloud lies in this handle's own zone outputs");
      zp = zone_params(h, pts, n_local, true, W);
      zp.mask_given = 0; zp.giant_plan = g->plan.get(); zp.giant_invalid_part = (uint32_t)me;
      zp.out_capacity = 0xFFFFFFF0u;  // nothing lands in the local outputs; the receivers' capacities are checked on the device
      CM_G_CUDA(g, cudaMemsetAsync(h->zw.overflow.get(), 0, sizeof(uint32_t), st));
      CM_G_CUDA(g, launch_zone_count_scan(zp, st));
      CM_G_CUDA(g, cudaMemcpyAsync(h->zw.zone_begin.get() + CM_MAX_ZONES + 1, g->p2p_words.get() + W + 1, sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
      h->zw.ran = false;  // no grouped array on this handle after this call
    } else {
      rc = zone_run(h, pts, n_local, st, true, W, g->plan.get(), (uint32_t)me);
      if (rc != CM_OK) return rc;
    }
    // every rank's per-destination offsets (NCCL takes the counts of a send / recv as host arguments)
    if (g->comm) CM_G_NCCL(g, g->api->AllGather(h->zw.zone_begin.get(), g->counts.get(), kCountStride, ncclUint32, g->comm, st));
    else CM_G_CUDA(g, cudaMemcpyAsync(g->counts.get() + (size_t)me * kCountStride, h->zw.zone_begin.get(), sizeof(uint32_t) * kCountStride, cudaMemcpyDeviceToDevice, st));
    CM_G_CUDA(g, cudaMemcpyAsync(g->counts_pin.get(), g->counts.get(), sizeof(uint32_t) * kCountStride * W, cudaMemcpyDeviceToHost, st));
    if (g->p2p) {
      CM_G_CUDA(g, launch_giant_offsets(g->counts.get(), kCountStride, (uint32_t)W, (uint32_t)me, g->p2p_words.get(), h->zw.overflow.get(), st));
      CM_G_CUDA(g, cudaMemcpyAsync(g->counts_pin.get() + (size_t)kCountStride * W, h->zw.overflow.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    }
  }
  CM_G_CUDA(g, cudaMemcpyAsync(g->plan_pin.get(), g->plan.get(), sizeof(GiantPlan), cudaMemcpyDeviceToHost, st));
  if (W > 1) CM_G_CUDA(g, mark(2));
  if (W > 1 && g->p2p) {
    CM_G_CUDA(g, cudaEventRecord(g->plan_ready.get(), st));
    for (int r = 0; r < W; ++r) zp.zone_ptr[r] = g->peer_recv[r];
    zp.zone_remote_base = g->p2p_words.get();
    CM_G_CUDA(g, launch_zone_scatter_remote(zp, st));
    // every store of every rank has landed once this one-word all-reduce completes (stream order on each rank)
    CM_G_NCCL(g, g->api->AllReduce(g->p2p_words.get() + W, g->p2p_words.get() + W, 1, ncclUint32, ncclMax, g->comm, st));
    CM_G_CUDA(g, cudaEventSynchronize(g->plan_ready.get()));  // the counts are here; the exchange is still in flight
  } else {
    CM_G_CUDA(g, cudaStreamSynchronize(st));
  }
  ++gi.host_syncs;
  const GiantPlan& P = *g->plan_pin;
  for (int k = 0; k < 3; ++k) {
    const uint32_t hi = f32_order_dec(P.enc[k]), lo = f32_order_dec(~P.enc[3 + k]);
    memcpy(&gi.max_p[k], &hi, 4); memcpy(&gi.min_p[k], &lo, 4);
    gi.min_b[k] = P.min_b[k]; gi.div_b[k] = P.div_b[k];
  }
  gi.key_bits = (int32_t)P.key_bits;
  // the histogram (and with it P.total) is only built for W > 1; one rank holds the whole cloud
  gi.points_total_finite = W > 1 ? (int64_t)P.total : n_local - (int64_t)P.n_invalid;
  for (int r = 0; r + 1 < W; ++r) gi.splitter[r] = P.splitter[r];
  if (P.error) return gfail(g, CM_E_KEY_RANGE, "the global voxel grid exceeds the key range (leaf too small for the extent)");
  const float4* vox_in = pts;
  int64_t n_vox = n_local;
  if (W > 1) {
    const uint32_t* mine = g->counts_pin.get() + (size_t)me * kCountStride;
    for (int r = 0; r <= W; ++r) gi.send_begin[r] = mine[r];
    gi.points_sent_away = n_local - (int64_t)(mine[me + 1] - mine[me]);
    if (!g->comm) {  // dry mode: the grouping is the result (cm_get_zone_out)
      if (info) *info = gi;
      return CM_OK;
    }
    int64_t roff[CM_MAX_ZONES + 1];
    roff[0] = 0;
    for (int s = 0; s < W; ++s) {
      const uint32_t* row = g->counts_pin.get() + (size_t)s * kCountStride;
      roff[s + 1] = roff[s] + (int64_t)(row[me + 1] - row[me]);
    }
    gi.points_received = roff[W];
    if (g->p2p) {
      // the device already decided (every rank the same): with an overflow nobody stored anything
      const uint32_t over = g->counts_pin.get()[(size_t)kCountStride * W];
      if (over) return gfail(g, CM_E_CAPACITY, "a rank would receive %u points, more than max_batch_points of its handle", over);
      gi.exchange = CM_GIANT_EXCHANGE_PEER;
      vox_in = g->recv.get();
      n_vox = roff[W];
    } else {
      if ((size_t)roff[W] > g->recv_cap)
        return gfail(g, CM_E_CAPACITY, "this rank receives %lld points, max_batch_points of the handle is %zu", (long long)roff[W], g->recv_cap);
      gi.exchange = CM_GIANT_EXCHANGE_NCCL;
      // ---- ONE all-to-all, straight out of the grouped array
      const float4* send = h->zw.out_xyzi.get();
      CM_G_NCCL(g, g->api->GroupStart());
      for (int r = 0; r < W; ++r) {
        const size_t sc = (size_t)(mine[r + 1] - mine[r]), rcnt = (size_t)(roff[r + 1] - roff[r]);
        if (r == me) continue;
        if (sc) CM_G_NCCL(g, g->api->Send(send + mine[r], sc * 4, ncclFloat, r, g->comm, st));
        if (rcnt) CM_G_NCCL(g, g->api->Recv(g->recv.get() + roff[r], rcnt * 4, ncclFloat, r, g->comm, st));
      }
      CM_G_NCCL(g, g->api->GroupEnd());
      const size_t self = (size_t)(mine[me + 1] - mine[me]);
      if (self) CM_G_CUDA(g, cudaMemcpyAsync(g->recv.get() + roff[me], send + mine[me], self * 16, cudaMemcpyDeviceToDevice, st));
      vox_in = g->recv.get();
      n_vox = roff[W];
    }
  } else {
    gi.points_received = n_local;
  }
  if (info) *info = gi;
  // ---- the ordinary single-GPU VoxelGrid on what arrived, global box folded in, key plan known from the global grid
  const uint32_t* enc_dev = reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(g->plan.get()) + offsetof(GiantPlan, enc));
  CM_G_CUDA(g, mark(3));
  // Non-finite points reach the local VoxelGrid only from this rank's own block (they are never sent away). k_grid_setup keys
  // them into a sentinel frame, which takes one more key bit: size the key and the pass count for it when there are any.
  rc = voxelgrid_run(h, vox_in, n_vox, st, enc_dev, (int)P.key_bits + (P.n_invalid ? 1 : 0));
  if (rc == CM_OK && prof && W > 1) {
    CM_G_CUDA(g, mark(4));
    CM_G_CUDA(g, cudaEventSynchronize(g->prof[4].get()));
    for (int i = 0; i < 4; ++i)
      if (cudaEventElapsedTime(&gi.stage_ms[i], g->prof[i].get(), g->prof[i + 1].get()) != cudaSuccess) { gi.stage_ms[i] = 0.f; cudaGetLastError(); }
    if (info) *info = gi;
  }
  return rc;
}

int cm_sync(cm_handle_t h) {
  if (!h) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  CM_CUDA(h, cudaSetDevice(h->device));
  if (!h->last) return fail(h, CM_E_INVALID, "nothing has run on this handle");
  return fetch_report(h, *h->last);
}

int cm_get_stats(cm_handle_t h, cm_stats_t* out) {
  if (!h || !out) return CM_E_INVALID;
  int rc = cm_sync(h);
  *out = h->stats;
  return rc;
}

int cm_get_device_out(cm_handle_t h, cm_device_out_t* out) {
  if (!h || !out) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!h->last || !h->last->has_run) return fail(h, CM_E_INVALID, "nothing has run on this handle");
  Workspace& w = *h->last;
  int rc = fetch_report(h, w);
  memset(out, 0, sizeof(*out));
  if (w.ran_k1) {
    int rc2 = materialize_dense(h, w);
    if (rc2 != CM_OK) return rc2;
    CM_CUDA(h, cudaStreamSynchronize(w.stream));
    out->survivor_xyzi = reinterpret_cast<const float*>(w.dense_xyzi.get());
    out->survivor_src = w.dense_src.get();
    out->survivor_slot = w.dense_slot.get();
    out->slot_xyzi = reinterpret_cast<const float*>(w.surv_xyzi.get());
  } else {
    out->survivor_xyzi = reinterpret_cast<const float*>(w.voxel_pts);
    out->slot_xyzi = out->survivor_xyzi;
  }
  if (w.ran_voxel) {
    const bool odd = (h->stats.sort_passes & 1) != 0;
    const SortInfo* si_rep = reinterpret_cast<const SortInfo*>(w.report.get() + w.ml.off_info);
    out->key_bytes = (int32_t)w.key_bytes;
    if (w.key_bytes == 4 && si_rep->segmented) {
      // a frame-segmented run sorted bare voxel indices: hand out (frame << idx_bits | idx), as every other run does,
      // in the ping-pong buffer the last pass did not write
      VoxelParams vp;
      fill_voxel_params(h, w, vp, w.voxel_pts, w.n_frames, (uint32_t)w.points_in);
      unsigned long long* k64 = reinterpret_cast<unsigned long long*>(odd ? w.keys_a.get() : w.keys_b.get());
      CM_CUDA(h, launch_seg_keys64(odd ? w.keys_b.get() : w.keys_a.get(), k64, w.vals_b.get(), vp, w.stream));
      CM_CUDA(h, cudaStreamSynchronize(w.stream));
      out->sorted_key = k64;
      out->sorted_point = w.vals_b.get();
      out->key_bytes = 8;
    } else if (w.key_bytes == 4) {
      // 32-bit keys are sorted as 8-byte (key, value) records: split them into the two arrays this struct promises
      const uint32_t* n_ptr = reinterpret_cast<const uint32_t*>(w.meta.get() + w.ml.off_fstart) + w.n_frames;
      VoxelParams vp;  // fused-key runs sorted box-grid keys: hand out PCL's index, like every other run
      fill_voxel_params(h, w, vp, w.voxel_pts, w.n_frames, (uint32_t)w.points_in);
      vp.fused_keys = w.fused_keys ? 1u : 0u;
      vp.box = w.box;
      CM_CUDA(h, launch_split_records(odd ? w.keys_b.get() : w.keys_a.get(), w.vals_a.get(), w.vals_b.get(), n_ptr, (uint32_t)w.points_in, w.stream,
                                      w.fused_keys ? &vp : nullptr));
      CM_CUDA(h, cudaStreamSynchronize(w.stream));
      out->sorted_key = w.vals_a.get();
      out->sorted_point = w.vals_b.get();
    } else {
      out->sorted_key = odd ? w.keys_b.get() : w.keys_a.get();
      out->sorted_point = odd ? w.vals_b.get() : w.vals_a.get();
    }
    out->voxel_xyzi = w.out_xyzi.get();
    out->voxel_count = w.out_count.get();
    out->voxel_idx = reinterpret_cast<const uint64_t*>(w.out_idx.get());
    out->key_idx_bits = (int32_t)si_rep->idx_bits;
  }
  return rc;
}

int cm_get_frame_info(cm_handle_t h, cm_frame_info_t* out, int capacity, int* n_frames) {
  if (!h) return CM_E_INVALID;
  int rc = cm_sync(h);
  std::lock_guard<std::mutex> lk(h->mu);
  const int n = (int)h->frame_info.size();
  if (n_frames) *n_frames = n;
  if (out) {
    if (capacity < n) return fail(h, CM_E_CAPACITY, "capacity %d < %d frames", capacity, n);
    for (int i = 0; i < n; ++i) out[i] = h->frame_info[i];
  }
  return rc;
}

int64_t cm_launch_count(cm_handle_t h) {
  if (!h || !h->last) return 0;
  return h->last->launches;
}

int cm_stage_ms(cm_handle_t h, const char* stage, float* ms) {
  if (!h || !stage || !ms) return CM_E_INVALID;
  int rc = cm_sync(h);
  int which = -1;
  if (!strcmp(stage, "total")) which = EV_START;
  else if (!strcmp(stage, "transform_crop")) which = EV_K1;
  else if (!strcmp(stage, "grid")) which = EV_GRID;
  else if (!strcmp(stage, "key_hist")) which = EV_KEY;
  else if (!strcmp(stage, "sort")) which = EV_SORT;
  else if (!strcmp(stage, "sort_pass0")) which = EV_SORT0;
  else if (!strcmp(stage, "centroid")) which = EV_CENT;
  if (which < 0) return fail(h, CM_E_INVALID, "unknown stage '%s'", stage);
  *ms = h->stage_ms[which];
  return rc;
}

int cm_debug_trace(cm_handle_t h, int which, uint64_t* out, int64_t capacity, int64_t* n) {
  if (!h || !n) return CM_E_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (!h->last) return fail(h, CM_E_INVALID, "nothing has run on this handle");
  Workspace& w = *h->last;
  const unsigned long long* src = which == 0 ? w.trace_k1.get() : w.trace_sort.get();
  const size_t cnt = which == 0 ? w.trace_k1_n : w.trace_sort_n;
  *n = (int64_t)cnt;
  if (!src) { *n = 0; return CM_OK; }
  if (!out) return CM_OK;
  if (capacity < (int64_t)cnt) return fail(h, CM_E_CAPACITY, "trace capacity");
  CM_CUDA(h, cudaSetDevice(h->device));
  CM_CUDA(h, cudaDeviceSynchronize());
  CM_CUDA(h, cudaMemcpy(out, src, cnt * 8, cudaMemcpyDeviceToHost));
  return CM_OK;
}

int cm_dev_alloc(cm_handle_t h, void** p, size_t bytes) {
  if (!h || !p) return CM_E_INVALID;
  CM_CUDA(h, cudaSetDevice(h->device));
  CM_CUDA(h, cudaMalloc(p, bytes ? bytes : 16));
  return CM_OK;
}
int cm_dev_free(cm_handle_t h, void* p) {
  if (!h) return CM_E_INVALID;
  CM_CUDA(h, cudaSetDevice(h->device));
  CM_CUDA(h, cudaFree(p));
  return CM_OK;
}
int cm_stream_create(cm_handle_t h, void** stream) {
  if (!h || !stream) return CM_E_INVALID;
  CM_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t st = nullptr;
  CM_CUDA(h, cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  *stream = st;
  return CM_OK;
}
int cm_stream_destroy(cm_handle_t h, void* stream) {
  if (!h) return CM_E_INVALID;
  CM_CUDA(h, cudaSetDevice(h->device));
  if (stream) CM_CUDA(h, cudaStreamDestroy(static_cast<cudaStream_t>(stream)));
  return CM_OK;
}
int cm_stream_sync(cm_handle_t h, void* stream) {
  if (!h) return CM_E_INVALID;
  CM_CUDA(h, cudaSetDevice(h->device));
  CM_CUDA(h, cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return CM_OK;
}
int cm_memcpy_h2d(cm_handle_t h, void* dst, const void* src, size_t bytes, void* stream) {
  if (!h) return CM_E_INVALID;
  CM_CUDA(h, cudaSetDevice(h->device));
  CM_CUDA(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)));
  CM_CUDA(h, cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return CM_OK;
}
int cm_memcpy_d2h(cm_handle_t h, void* dst, const void* src, size_t bytes, void* stream) {
  if (!h) return CM_E_INVALID;
  CM_CUDA(h, cudaSetDevice(h->device));
  CM_CUDA(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)));
  CM_CUDA(h, cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return CM_OK;
}

}  // extern "C"
