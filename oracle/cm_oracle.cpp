/*
 * cm_oracle.cpp -- CPU oracle for the cloud_merger merge hot path (TEST INFRASTRUCTURE ONLY; see cm_oracle.h).
 *
 * PARITY UNPINNED (no reference tests / golden vectors exist; PCL 1.8.1, pcl_ros 1.7 and Eigen 3.3.4 are absent from
 * /root/reference and from this image). Restatement of the published PCL 1.8.1 algorithms, anchored on the reference
 * call sites cited at each function.
 *
 * Build: g++ -O2 -std=c++17 -ffp-contract=off -fPIC -shared -pthread (oracle/Makefile). No -march, no -ffast-math: the
 * reference is compiled for baseline x86-64, so every float multiply and add below rounds on its own.
 */
#include "cm_oracle.h"

#include <algorithm>
#include <array>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <limits>
#include <thread>
#include <vector>

namespace {

/* pcl::PointXYZI: 32 bytes, 16-byte aligned; data[3] = 1.0f; intensity at byte 16 (PCL point_types.hpp). */
struct alignas(16) PointXYZI {
  float x, y, z, pad;
  float intensity, c1, c2, c3;
  PointXYZI() : x(0.f), y(0.f), z(0.f), pad(1.f), intensity(0.f), c1(0.f), c2(0.f), c3(0.f) {}
};
static_assert(sizeof(PointXYZI) == 32, "PointXYZI layout");

/* The members of pcl::PointCloud<PointXYZI> the path touches. */
struct Cloud {
  std::vector<PointXYZI> points;
  uint32_t width = 0, height = 0;
  bool is_dense = true;
  uint64_t stamp = 0;
};

inline bool finite3(const PointXYZI& p) { return std::isfinite(p.x) && std::isfinite(p.y) && std::isfinite(p.z); }

inline float load_f32(const uint8_t* p) {
  float v;
  std::memcpy(&v, p, sizeof(float));
  return v;
}

/* a1 -- pcl_ros/point_cloud.h Serializer<pcl::PointCloud<T>>::read via pcl::createMapping: fields matched by name
 * (x, y, z, intensity; FLOAT32) and copied into the PointXYZI record. Reference: the subscribers at
 * pc_preprocessing_main.cpp:520-525 and CloudFusionNode.h:51-56. */
void unpack_cloud(const uint8_t* data, int64_t n, int step, int ox, int oy, int oz, int oi, Cloud& out) {
  out.points.resize(static_cast<size_t>(n));
  for (int64_t i = 0; i < n; ++i) {
    const uint8_t* rec = data + i * static_cast<int64_t>(step);
    PointXYZI& p = out.points[static_cast<size_t>(i)];
    p.x = load_f32(rec + ox);
    p.y = load_f32(rec + oy);
    p.z = load_f32(rec + oz);
    p.intensity = oi >= 0 ? load_f32(rec + oi) : 0.f;
  }
  out.width = static_cast<uint32_t>(n);
  out.height = 1;
}

/* a2 -- pcl::transformPointCloud(cloud_in, cloud_out, Eigen::Affine3f) of PCL 1.8.1 (common/impl/transforms.hpp), which is
 * what pcl_ros::transformPointCloud(in, out, tf::Transform) ends in. Reference call sites:
 * pc_preprocessing_main.cpp:322,348,373,399,426,465; CloudFusionNode.h:508-533.
 * x' = ((m00*x + m01*y) + m02*z) + m03, left to right, unfused. A non-dense cloud keeps non-finite points unchanged. */
void transform_cloud(const Cloud& in, Cloud& out, const float* m) {
  if (&in != &out) {
    out.points.assign(in.points.begin(), in.points.end()); /* the reference copies the whole cloud first */
    out.width = in.width;
    out.height = in.height;
    out.is_dense = in.is_dense;
    out.stamp = in.stamp;
  }
  const size_t n = out.points.size();
  for (size_t i = 0; i < n; ++i) {
    const float x = in.points[i].x, y = in.points[i].y, z = in.points[i].z;
    if (!in.is_dense && !(std::isfinite(x) && std::isfinite(y) && std::isfinite(z))) continue;
    const float nx = ((m[0] * x + m[1] * y) + m[2] * z) + m[3];
    const float ny = ((m[4] * x + m[5] * y) + m[6] * z) + m[7];
    const float nz = ((m[8] * x + m[9] * y) + m[10] * z) + m[11];
    out.points[i].x = nx;
    out.points[i].y = ny;
    out.points[i].z = nz;
  }
}

inline float field_of(const PointXYZI& p, int axis) {
  switch (axis) {
    case 0: return p.x;
    case 1: return p.y;
    case 2: return p.z;
    default: return p.intensity;
  }
}

/* a3..a6 -- pcl::PassThrough<PointT>::applyFilterIndices of PCL 1.8.1 (filters/impl/passthrough.hpp): limits are float,
 * the window is inclusive, non-finite xyz or a non-finite field value is always removed, order is kept.
 * Reference: getROI pc_preprocessing_main.cpp:20-40, getCloudPart :49-59, removeGround :80-92,
 * filter_ROI_R CloudFusionNode.h:145-190, remove_ground :201-216. */
void passthrough_indices(const Cloud& in, int axis, float lo, float hi, bool negative, std::vector<int>& indices) {
  indices.resize(in.points.size());
  size_t oii = 0;
  for (size_t iii = 0; iii < in.points.size(); ++iii) {
    const PointXYZI& p = in.points[iii];
    if (!finite3(p)) continue;
    const float v = field_of(p, axis);
    if (!std::isfinite(v)) continue;
    if (!negative && (v < lo || v > hi)) continue;
    if (negative && v >= lo && v <= hi) continue;
    indices[oii++] = static_cast<int>(iii);
  }
  indices.resize(oii);
}

/* pcl::copyPointCloud(cloud_in, indices, cloud_out): what Filter::filter does with the kept indices. */
void copy_by_indices(const Cloud& in, const std::vector<int>& indices, Cloud& out) {
  std::vector<PointXYZI> pts(indices.size());
  for (size_t i = 0; i < indices.size(); ++i) pts[i] = in.points[static_cast<size_t>(indices[i])];
  out.points.swap(pts);
  out.width = static_cast<uint32_t>(out.points.size());
  out.height = 1;
  out.is_dense = true; /* PassThrough output is clean */
  out.stamp = in.stamp;
}

/* a7 -- pcl::PointCloud<PointT>::operator+= of PCL 1.8.1 (common/include/pcl/point_cloud.h).
 * Reference: fusePointclouds pc_preprocessing_main.cpp:137-149, cloud_fusion CloudFusionNode.h:64-69. */
void concat_into(Cloud& lhs, const Cloud& rhs) {
  if (rhs.stamp > lhs.stamp) lhs.stamp = rhs.stamp;
  const size_t nr = lhs.points.size();
  lhs.points.resize(nr + rhs.points.size());
  for (size_t i = nr; i < lhs.points.size(); ++i) lhs.points[i] = rhs.points[i - nr];
  lhs.width = static_cast<uint32_t>(lhs.points.size());
  lhs.height = 1;
  lhs.is_dense = rhs.is_dense && lhs.is_dense;
}

struct IndexPair32 {
  unsigned int idx;
  unsigned int cloud_point_index;
  bool operator<(const IndexPair32& o) const { return idx < o.idx; }
};
struct IndexPair64 {
  int64_t idx;
  unsigned int cloud_point_index;
  bool operator<(const IndexPair64& o) const { return idx < o.idx; }
};

struct VoxelOut {
  float* xyzi;       /* float sums, ascending point index */
  float* xyzi_sort;  /* float sums, std::sort order */
  double* xyzi_f64;  /* double sums, ascending point index */
  uint32_t* count;
  int64_t* idx;
  int64_t* point_idx;
  int32_t* grid;
  int32_t* flags;
};

template <typename Pair>
int64_t voxel_runs(const Cloud& in, std::vector<Pair>& iv, uint32_t min_points, bool downsample_all, const VoxelOut& o) {
  /* Second pass: sort by target cell (std::sort: unstable, as in PCL). */
  std::sort(iv.begin(), iv.end());
  /* Third pass: runs of equal idx, dropped when shorter than min_points_per_voxel_. */
  std::vector<std::pair<unsigned int, unsigned int>> fl;
  fl.reserve(iv.size());
  unsigned int index = 0;
  while (index < iv.size()) {
    unsigned int i = index + 1;
    while (i < iv.size() && iv[i].idx == iv[index].idx) ++i;
    if (i - index >= min_points) fl.emplace_back(index, i);
    index = i;
  }
  /* Fourth pass: centroids (pcl::CentroidPoint<PointXYZI>: AccumulatorXYZ = Vector3f sum / n, AccumulatorIntensity =
   * float sum / n; with downsample_all_data_ == false only xyz is averaged and intensity stays default 0). */
  std::vector<unsigned int> members;
  for (size_t cp = 0; cp < fl.size(); ++cp) {
    const unsigned int first = fl[cp].first, last = fl[cp].second;
    const float nf = static_cast<float>(last - first);
    if (o.xyzi_sort) {
      float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
      for (unsigned int li = first; li < last; ++li) {
        const PointXYZI& p = in.points[iv[li].cloud_point_index];
        sx += p.x; sy += p.y; sz += p.z; si += p.intensity;
      }
      o.xyzi_sort[cp * 4 + 0] = sx / nf;
      o.xyzi_sort[cp * 4 + 1] = sy / nf;
      o.xyzi_sort[cp * 4 + 2] = sz / nf;
      o.xyzi_sort[cp * 4 + 3] = downsample_all ? si / nf : 0.f;
    }
    if (o.xyzi || o.xyzi_f64) {
      members.clear();
      for (unsigned int li = first; li < last; ++li) members.push_back(iv[li].cloud_point_index);
      std::sort(members.begin(), members.end());
      float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
      double dx = 0., dy = 0., dz = 0., di = 0.;
      for (unsigned int pi : members) {
        const PointXYZI& p = in.points[pi];
        sx += p.x; sy += p.y; sz += p.z; si += p.intensity;
        dx += p.x; dy += p.y; dz += p.z; di += p.intensity;
      }
      if (o.xyzi) {
        o.xyzi[cp * 4 + 0] = sx / nf;
        o.xyzi[cp * 4 + 1] = sy / nf;
        o.xyzi[cp * 4 + 2] = sz / nf;
        o.xyzi[cp * 4 + 3] = downsample_all ? si / nf : 0.f;
      }
      if (o.xyzi_f64) {
        const double nd = static_cast<double>(last - first);
        o.xyzi_f64[cp * 4 + 0] = dx / nd;
        o.xyzi_f64[cp * 4 + 1] = dy / nd;
        o.xyzi_f64[cp * 4 + 2] = dz / nd;
        o.xyzi_f64[cp * 4 + 3] = downsample_all ? di / nd : 0.;
      }
    }
    if (o.count) o.count[cp] = last - first;
    if (o.idx) o.idx[cp] = static_cast<int64_t>(iv[first].idx);
  }
  return static_cast<int64_t>(fl.size());
}

/* a8 -- pcl::VoxelGrid<PointT>::applyFilter of PCL 1.8.1 (filters/impl/voxel_grid.hpp), no filter field.
 * Reference: voxelgrid pc_preprocessing_main.cpp:168-177, CloudFusionNode.h:276-289, PreprocessingNode.h:236-249. */
int64_t voxelgrid_cloud(const Cloud& in, const float* leaf, uint32_t min_points, bool downsample_all, bool force64,
                        const VoxelOut& o) {
  if (o.flags) *o.flags = 0;
  const size_t n = in.points.size();
  if (o.point_idx)
    for (size_t i = 0; i < n; ++i) o.point_idx[i] = -1;
  if (o.grid)
    for (int k = 0; k < 9; ++k) o.grid[k] = 0;
  if (n == 0) return 0;

  /* inverse_leaf_size_ = Array4f::Ones() / leaf_size_.array() */
  const float inv[3] = {1.0f / leaf[0], 1.0f / leaf[1], 1.0f / leaf[2]};

  /* pcl::getMinMax3D(cloud, indices, min_p, max_p): non-finite points are skipped only when !is_dense. The oracle also
   * skips them for a cloud flagged dense (PCL's result is undefined there; the build defines it this way). */
  float min_p[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, max_p[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  size_t n_valid = 0;
  for (size_t i = 0; i < n; ++i) {
    const PointXYZI& p = in.points[i];
    if (!finite3(p)) continue;
    ++n_valid;
    min_p[0] = std::min(min_p[0], p.x); max_p[0] = std::max(max_p[0], p.x);
    min_p[1] = std::min(min_p[1], p.y); max_p[1] = std::max(max_p[1], p.y);
    min_p[2] = std::min(min_p[2], p.z); max_p[2] = std::max(max_p[2], p.z);
  }
  if (n_valid == 0) return 0;

  /* "Check that the leaf size is not too small, given the size of the data" */
  const int64_t dx = static_cast<int64_t>((max_p[0] - min_p[0]) * inv[0]) + 1;
  const int64_t dy = static_cast<int64_t>((max_p[1] - min_p[1]) * inv[1]) + 1;
  const int64_t dz = static_cast<int64_t>((max_p[2] - min_p[2]) * inv[2]) + 1;
  // PCL writes (dx * dy * dz) > INT32_MAX in int64_t, which overflows (undefined) from 2^63 on -- 2^21 cells on every axis.
  // The product is compared step by step so that every partial product stays below 2^62: the guard trips as it does
  // mathematically (np_oracle compares the exact product).
  const int64_t imax = static_cast<int64_t>(std::numeric_limits<int32_t>::max());
  const bool pcl_overflow = dx > imax || dy > imax || dz > imax || dx < 0 || dy < 0 || dz < 0 || dx * dy > imax ||
                            dx * dy * dz > imax;
  if (pcl_overflow) {
    if (o.flags) *o.flags |= CMO_FLAG_PCL_OVERFLOW;
    if (!force64) { /* PCL: PCL_WARN(...); output = *input_; return; */
      if (o.xyzi)
        for (size_t i = 0; i < n; ++i) {
          o.xyzi[i * 4 + 0] = in.points[i].x; o.xyzi[i * 4 + 1] = in.points[i].y;
          o.xyzi[i * 4 + 2] = in.points[i].z; o.xyzi[i * 4 + 3] = in.points[i].intensity;
        }
      return static_cast<int64_t>(n);
    }
  }

  int64_t min_b[3], max_b[3], div_b[3];
  for (int a = 0; a < 3; ++a) {
    min_b[a] = static_cast<int64_t>(std::floor(min_p[a] * inv[a]));
    max_b[a] = static_cast<int64_t>(std::floor(max_p[a] * inv[a]));
    div_b[a] = max_b[a] - min_b[a] + 1;
  }
  if (o.grid)
    for (int a = 0; a < 3; ++a) {
      o.grid[a] = static_cast<int32_t>(min_b[a]);
      o.grid[3 + a] = static_cast<int32_t>(max_b[a]);
      o.grid[6 + a] = static_cast<int32_t>(div_b[a]);
    }

  if (!force64) {
    /* PCL's own int32 formulation. divb_mul_ = (1, div0, div0*div1). */
    const int div0 = static_cast<int>(div_b[0]), div1 = static_cast<int>(div_b[1]);
    const int mul1 = div0, mul2 = div0 * div1;
    const int mb0 = static_cast<int>(min_b[0]), mb1 = static_cast<int>(min_b[1]), mb2 = static_cast<int>(min_b[2]);
    std::vector<IndexPair32> iv;
    iv.reserve(n);
    for (size_t i = 0; i < n; ++i) {
      const PointXYZI& p = in.points[i];
      if (!finite3(p)) continue;
      const int ijk0 = static_cast<int>(std::floor(p.x * inv[0]) - static_cast<float>(mb0));
      const int ijk1 = static_cast<int>(std::floor(p.y * inv[1]) - static_cast<float>(mb1));
      const int ijk2 = static_cast<int>(std::floor(p.z * inv[2]) - static_cast<float>(mb2));
      const int idx = ijk0 + ijk1 * mul1 + ijk2 * mul2;
      iv.push_back({static_cast<unsigned int>(idx), static_cast<unsigned int>(i)});
      if (o.point_idx) o.point_idx[i] = static_cast<int64_t>(static_cast<unsigned int>(idx));
    }
    return voxel_runs(in, iv, min_points, downsample_all, o);
  }
  /* 64-bit extension: the same linearisation in int64 (identical to the int32 one wherever PCL accepts the cloud). */
  const int64_t mul1 = div_b[0], mul2 = div_b[0] * div_b[1];
  std::vector<IndexPair64> iv;
  iv.reserve(n);
  for (size_t i = 0; i < n; ++i) {
    const PointXYZI& p = in.points[i];
    if (!finite3(p)) continue;
    const int64_t ijk0 = static_cast<int64_t>(std::floor(p.x * inv[0])) - min_b[0];
    const int64_t ijk1 = static_cast<int64_t>(std::floor(p.y * inv[1])) - min_b[1];
    const int64_t ijk2 = static_cast<int64_t>(std::floor(p.z * inv[2])) - min_b[2];
    const int64_t idx = ijk0 + ijk1 * mul1 + ijk2 * mul2;
    iv.push_back({idx, static_cast<unsigned int>(i)});
    if (o.point_idx) o.point_idx[i] = idx;
  }
  return voxel_runs(in, iv, min_points, downsample_all, o);
}

void cloud_from_xyzi(const float* xyzi, int64_t n, bool is_dense, Cloud& c) {
  c.points.resize(static_cast<size_t>(n));
  for (int64_t i = 0; i < n; ++i) {
    PointXYZI& p = c.points[static_cast<size_t>(i)];
    p.x = xyzi[i * 4 + 0]; p.y = xyzi[i * 4 + 1]; p.z = xyzi[i * 4 + 2]; p.intensity = xyzi[i * 4 + 3];
  }
  c.width = static_cast<uint32_t>(n);
  c.height = 1;
  c.is_dense = is_dense;
}

/* One sensor callback up to the end of the crop chain: callbackX -> transformPointCloud -> getROI/getCloudPart style
 * PassThrough chain (pc_preprocessing_main.cpp:318-337, :20-59). Every pass copies its survivors into a new cloud, as the
 * reference's filter(*cloud_ROI_ptr) does. kept[] receives, per surviving point, its index in the sensor's input. */
void sensor_path(const cmo_cloud_t& c, const cmo_pass_t* passes, int n_passes, Cloud& out, std::vector<uint32_t>& kept) {
  Cloud raw;
  unpack_cloud(c.data, c.n_points, c.point_step, c.off_x, c.off_y, c.off_z, c.off_i, raw);
  raw.is_dense = c.is_dense != 0;
  Cloud cur;
  transform_cloud(raw, cur, c.m);
  kept.resize(cur.points.size());
  for (size_t i = 0; i < kept.size(); ++i) kept[i] = static_cast<uint32_t>(i);
  std::vector<int> idx;
  std::vector<uint32_t> kept2;
  for (int k = 0; k < n_passes; ++k) {
    passthrough_indices(cur, passes[k].axis, passes[k].lo, passes[k].hi, passes[k].negative != 0, idx);
    kept2.resize(idx.size());
    for (size_t i = 0; i < idx.size(); ++i) kept2[i] = kept[static_cast<size_t>(idx[i])];
    kept.swap(kept2);
    copy_by_indices(cur, idx, cur);
  }
  out.points.swap(cur.points);
  out.width = static_cast<uint32_t>(out.points.size());
  out.height = 1;
  out.is_dense = cur.is_dense;
}

}  // namespace

extern "C" {

void cmo_unpack(const uint8_t* data, int64_t n, int32_t point_step, int32_t off_x, int32_t off_y, int32_t off_z,
                int32_t off_i, float* out_xyzi) {
  Cloud c;
  unpack_cloud(data, n, point_step, off_x, off_y, off_z, off_i, c);
  for (int64_t i = 0; i < n; ++i) {
    const PointXYZI& p = c.points[static_cast<size_t>(i)];
    out_xyzi[i * 4 + 0] = p.x; out_xyzi[i * 4 + 1] = p.y; out_xyzi[i * 4 + 2] = p.z; out_xyzi[i * 4 + 3] = p.intensity;
  }
}

void cmo_transform(const float* in_xyzi, int64_t n, const float* m, int32_t is_dense, float* out_xyzi) {
  Cloud in, out;
  cloud_from_xyzi(in_xyzi, n, is_dense != 0, in);
  transform_cloud(in, out, m);
  for (int64_t i = 0; i < n; ++i) {
    const PointXYZI& p = out.points[static_cast<size_t>(i)];
    out_xyzi[i * 4 + 0] = p.x; out_xyzi[i * 4 + 1] = p.y; out_xyzi[i * 4 + 2] = p.z; out_xyzi[i * 4 + 3] = p.intensity;
  }
}

int64_t cmo_passthrough(const float* in_xyzi, int64_t n, int32_t axis, float lo, float hi, int32_t negative,
                        int32_t* out_indices) {
  Cloud in;
  cloud_from_xyzi(in_xyzi, n, true, in);
  std::vector<int> idx;
  passthrough_indices(in, axis, lo, hi, negative != 0, idx);
  for (size_t i = 0; i < idx.size(); ++i) out_indices[i] = idx[i];
  return static_cast<int64_t>(idx.size());
}

int64_t cmo_voxelgrid(const float* xyzi, int64_t n, int32_t is_dense, const float* leaf, uint32_t min_points,
                      int32_t downsample_all, int32_t force64, float* out_xyzi, float* out_xyzi_sort,
                      double* out_xyzi_f64, uint32_t* out_count, int64_t* out_idx, int64_t* point_idx, int32_t* grid,
                      int32_t* flags) {
  Cloud in;
  cloud_from_xyzi(xyzi, n, is_dense != 0, in);
  VoxelOut o{out_xyzi, out_xyzi_sort, out_xyzi_f64, out_count, out_idx, point_idx, grid, flags};
  return voxelgrid_cloud(in, leaf, min_points, downsample_all != 0, force64 != 0, o);
}

int64_t cmo_merge_frame(const cmo_cloud_t* clouds, int32_t n_clouds, const cmo_pass_t* passes, int32_t n_passes,
                        const float* leaf, uint32_t min_points, int32_t downsample_all, int32_t force64,
                        int32_t threads, float* out_survivor_xyzi, uint32_t* out_survivor_src, int64_t* n_survivors,
                        float* out_xyzi, double* out_xyzi_f64, uint32_t* out_count, int64_t* out_idx,
                        int64_t* point_idx, int32_t* grid, int32_t* flags) {
  std::vector<Cloud> per(static_cast<size_t>(n_clouds));
  std::vector<std::vector<uint32_t>> kept(static_cast<size_t>(n_clouds));
  if (threads <= 1) {
    for (int s = 0; s < n_clouds; ++s) sensor_path(clouds[s], passes, n_passes, per[s], kept[s]);
  } else {
    /* the reference runs the sensor callbacks on ros::AsyncSpinner(6) threads (pc_preprocessing_main.cpp:513) */
    std::vector<std::thread> pool;
    const int nt = std::min<int>(threads, n_clouds);
    for (int t = 0; t < nt; ++t)
      pool.emplace_back([&, t]() {
        for (int s = t; s < n_clouds; s += nt) sensor_path(clouds[s], passes, n_passes, per[s], kept[s]);
      });
    for (auto& th : pool) th.join();
  }
  /* fusePointclouds (pc_preprocessing_main.cpp:137-142): assign the first, += the rest, sensor order. */
  Cloud fused;
  std::vector<uint32_t> src;
  uint32_t base = 0;
  for (int s = 0; s < n_clouds; ++s) {
    if (s == 0) fused = per[0]; else concat_into(fused, per[s]);
    for (uint32_t k : kept[s]) src.push_back(base + k);
    base += static_cast<uint32_t>(clouds[s].n_points);
  }
  const size_t m = fused.points.size();
  if (n_survivors) *n_survivors = static_cast<int64_t>(m);
  if (out_survivor_xyzi)
    for (size_t i = 0; i < m; ++i) {
      const PointXYZI& p = fused.points[i];
      out_survivor_xyzi[i * 4 + 0] = p.x; out_survivor_xyzi[i * 4 + 1] = p.y;
      out_survivor_xyzi[i * 4 + 2] = p.z; out_survivor_xyzi[i * 4 + 3] = p.intensity;
    }
  if (out_survivor_src)
    for (size_t i = 0; i < m; ++i) out_survivor_src[i] = src[i];
  /* voxelgrid (pc_preprocessing_main.cpp:168-177) */
  VoxelOut o{out_xyzi, nullptr, out_xyzi_f64, out_count, out_idx, point_idx, grid, flags};
  return voxelgrid_cloud(fused, leaf, min_points, downsample_all != 0, force64 != 0, o);
}

void cmo_tf_to_matrix(const double* q, const double* t, float* m) {
  /* pcl_ros::transformPointCloud: Eigen::Quaternionf rotation(q.w, q.x, q.y, q.z); Eigen::Vector3f origin(v);
   * Affine3f t(Translation3f(origin) * rotation). Eigen 3.3.4 QuaternionBase::toRotationMatrix. */
  const float x = static_cast<float>(q[0]), y = static_cast<float>(q[1]), z = static_cast<float>(q[2]),
              w = static_cast<float>(q[3]);
  const float tx = 2.0f * x, ty = 2.0f * y, tz = 2.0f * z;
  const float twx = tx * w, twy = ty * w, twz = tz * w;
  const float txx = tx * x, txy = ty * x, txz = tz * x;
  const float tyy = ty * y, tyz = tz * y, tzz = tz * z;
  m[0] = 1.0f - (tyy + tzz); m[1] = txy - twz;          m[2] = txz + twy;           m[3] = static_cast<float>(t[0]);
  m[4] = txy + twz;          m[5] = 1.0f - (txx + tzz); m[6] = tyz - twx;           m[7] = static_cast<float>(t[1]);
  m[8] = txz - twy;          m[9] = tyz + twx;          m[10] = 1.0f - (txx + tyy); m[11] = static_cast<float>(t[2]);
}

/* pcl::RadiusOutlierRemoval<PointXYZI>::applyFilterIndices of PCL 1.8.1 (filters/impl/radius_outlier_removal.hpp), as
 * configured by the reference's outlierRemoval() (pc_preprocessing_main.cpp:184-192: setRadiusSearch(radius),
 * setMinNeighborsInRadius(min_neighbor), keep_organized false; Parameter.h:23-24 radius 0.15, min_neighbor 1):
 *   k = searcher_->radiusSearch(point, search_radius_, ...)   -- k counts the query point itself
 *   outlier  <=>  (!negative && k <= min_pts) || (negative && k > min_pts)
 * The search is pcl::search::KdTree -> pcl::KdTreeFLANN (FLANN 1.8/1.9, L2_Simple<float>): a point is inside the radius
 * iff its squared distance, accumulated in float as ((0 + dx*dx) + dy*dy) + dz*dz with dx = query - data, is strictly
 * smaller than (float)(radius * radius) (radius is a double in PCL; RadiusResultSet::addPoint tests dist < radius).
 * The kd-tree only prunes; it does not change which points are counted, so an exhaustive count over a cell grid whose
 * cells are two radii wide gives the same k. Non-finite points are never kept (PCL requires a dense cloud here; the
 * reference applies the filter to PassThrough/ExtractIndices output, which is dense).
 * Writes the indices of the kept points in input order; returns how many. */
int64_t cmo_radius_outlier(const float* xyzi, int64_t n, double radius, int32_t min_pts, int32_t negative,
                           int32_t* out_indices) {
  const float r2 = static_cast<float>(radius * radius);
  const double cell = radius > 0.0 ? 2.0 * radius : 1.0;
  /* grid over the finite points (double arithmetic: only a pruning structure, with a full cell of slack) */
  std::vector<int64_t> order;
  std::vector<std::array<int64_t, 3>> cell_of(static_cast<size_t>(n));
  std::vector<char> fin(static_cast<size_t>(n), 0);
  for (int64_t i = 0; i < n; ++i) {
    const float* p = xyzi + i * 4;
    if (std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2])) {
      fin[i] = 1;
      for (int a = 0; a < 3; ++a) cell_of[i][a] = static_cast<int64_t>(std::floor(static_cast<double>(p[a]) / cell));
      order.push_back(i);
    }
  }
  std::sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
    if (cell_of[a] != cell_of[b]) return cell_of[a] < cell_of[b];
    return a < b;
  });
  auto find_cell = [&](const std::array<int64_t, 3>& c) {
    return std::lower_bound(order.begin(), order.end(), c,
                            [&](int64_t idx, const std::array<int64_t, 3>& key) { return cell_of[idx] < key; });
  };
  int64_t kept = 0;
  for (int64_t i = 0; i < n; ++i) {
    if (!fin[i]) continue;
    const float* q = xyzi + i * 4;
    int64_t k = 0;
    for (int64_t dz = -1; dz <= 1; ++dz)
      for (int64_t dy = -1; dy <= 1; ++dy)
        for (int64_t dx = -1; dx <= 1; ++dx) {
          const std::array<int64_t, 3> c = {cell_of[i][0] + dx, cell_of[i][1] + dy, cell_of[i][2] + dz};
          for (auto it = find_cell(c); it != order.end() && cell_of[*it] == c; ++it) {
            const float* d = xyzi + (*it) * 4;
            float acc = 0.0f;
            for (int a = 0; a < 3; ++a) {
              const float diff = q[a] - d[a];
              acc += diff * diff;
            }
            if (acc < r2) ++k;
          }
        }
    const bool outlier = (!negative && k <= min_pts) || (negative && k > min_pts);
    if (!outlier) out_indices[kept++] = static_cast<int32_t>(i);
  }
  return kept;
}

/* ---- RANSAC ground plane: pcl::SACSegmentation<PointXYZI> with SACMODEL_PLANE / SAC_RANSAC --------------------------
 * Reference call site: pc_preprocessing_main.cpp:95-117 (setOptimizeCoefficients(true), setMaxIterations(1000),
 * setDistanceThreshold(0.3f), setProbability(0.99f); setAxis / setEpsAngle are set there but SACMODEL_PLANE ignores
 * them), followed by pcl::ExtractIndices with the inliers (negative and positive). Parameters: Parameter.h:38-42.
 * Restated from PCL 1.8.1 (sample_consensus/{sac_model.h, impl/sac_model_plane.hpp, impl/ransac.hpp},
 * segmentation/impl/sac_segmentation.hpp, common/impl/{centroid,eigen}.hpp), Eigen 3.3.4 and Boost.Random:
 *
 *  sampler   SampleConsensusModel with random == false seeds boost::mt19937 with 12345 and draws through
 *            boost::uniform_int<>(0, INT_MAX), which maps the 32-bit engine output to out >> 1. drawIndexSample swaps
 *            shuffled_indices_[i] with shuffled_indices_[i + rnd() % (n - i)] for i = 0, 1, 2 (the array persists over
 *            the draws of one segment() call) and takes the first three entries. getSamples repeats the draw (at most
 *            max_sample_checks_ = 1000 times) until isSampleGood: ((p1-p0)/(p2-p0)) has unequal x, y, z quotients.
 *  model     cross product of (p1-p0) and (p2-p0), Eigen 3.3 normalize() (divides by sqrt(squaredNorm) iff that is > 0),
 *            d = -1 * dot(n, p0).
 *  score     countWithinDistance: |dot((a,b,c,d), (x,y,z,1))| < threshold, strict.
 *  loop      RandomSampleConsensus::computeModel: k = log(1 - p) / log(1 - w^3) is lowered at every new best model,
 *            the loop ends when iterations >= k or iterations > max_iterations.
 *  refine    optimizeModelCoefficients: float running sums of xx, xy, xz, yy, yz, zz, x, y, z over the inliers in index
 *            order, / n, covariance = E[ab] - E[a]E[b], pcl::eigen33 (closed-form smallest eigenvalue in float, eigenvector
 *            from the largest row cross product), d = -1 * dot(n, centroid); then selectWithinDistance once more.
 *
 * The 4-wide float dot products / squared norms are Eigen packet reductions whose order depends on the instruction set
 * PCL was built for; sum_order selects it: 0 = SSE2 (movehl + shuffle): (l0+l2)+(l1+l3); 1 = SSE3 (haddps):
 * (l0+l1)+(l2+l3); 2 = scalar: ((l0+l1)+l2)+l3. */
namespace {
struct Mt19937 {
  uint32_t s[624];
  int at;
  explicit Mt19937(uint32_t seed) {
    s[0] = seed;
    for (int i = 1; i < 624; ++i) s[i] = 1812433253u * (s[i - 1] ^ (s[i - 1] >> 30)) + static_cast<uint32_t>(i);
    at = 624;
  }
  void refill() {
    for (int i = 0; i < 624; ++i) {
      const uint32_t y = (s[i] & 0x80000000u) | (s[(i + 1) % 624] & 0x7fffffffu);
      s[i] = s[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    at = 0;
  }
  uint32_t next() {
    if (at >= 624) refill();
    uint32_t y = s[at++];
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
  }
};

inline float sum4(float l0, float l1, float l2, float l3, int order) {
  if (order == 0) return (l0 + l2) + (l1 + l3);
  if (order == 1) return (l0 + l1) + (l2 + l3);
  return ((l0 + l1) + l2) + l3;
}

inline bool plane_sample_good(const float* p0, const float* p1, const float* p2) {
  float q[3];
  for (int a = 0; a < 3; ++a) q[a] = (p1[a] - p0[a]) / (p2[a] - p0[a]);
  return (q[0] != q[1]) || (q[2] != q[1]);
}

inline void plane_from_sample(const float* p0, const float* p1, const float* p2, int order, float* c) {
  float u[3], v[3];
  for (int a = 0; a < 3; ++a) { u[a] = p1[a] - p0[a]; v[a] = p2[a] - p0[a]; }
  c[0] = u[1] * v[2] - u[2] * v[1];
  c[1] = u[2] * v[0] - u[0] * v[2];
  c[2] = u[0] * v[1] - u[1] * v[0];
  c[3] = 0.0f;
  const float z = sum4(c[0] * c[0], c[1] * c[1], c[2] * c[2], c[3] * c[3], order);
  if (z > 0.0f) {
    const float nrm = std::sqrt(z);
    for (int a = 0; a < 4; ++a) c[a] = c[a] / nrm;
  }
  c[3] = -1.0f * sum4(c[0] * p0[0], c[1] * p0[1], c[2] * p0[2], c[3] * 1.0f, order);
}

inline float plane_distance(const float* c, const float* p, int order) {
  return std::fabs(sum4(c[0] * p[0], c[1] * p[1], c[2] * p[2], c[3] * 1.0f, order));
}

/* pcl::computeRoots2 / computeRoots / eigen33 (smallest eigenvalue form), Scalar = float */
void roots2(float b, float c, float* r) {
  r[0] = 0.0f;
  float d = static_cast<float>(b * b - 4.0 * c);
  if (d < 0.0) d = 0.0f;
  const float sd = std::sqrt(d);
  r[2] = 0.5f * (b + sd);
  r[1] = 0.5f * (b - sd);
}

void roots3(const float m[3][3], float* r) {
  const float c0 = m[0][0] * m[1][1] * m[2][2] + 2.0f * m[0][1] * m[0][2] * m[1][2] - m[0][0] * m[1][2] * m[1][2] -
                   m[1][1] * m[0][2] * m[0][2] - m[2][2] * m[0][1] * m[0][1];
  const float c1 = m[0][0] * m[1][1] - m[0][1] * m[0][1] + m[0][0] * m[2][2] - m[0][2] * m[0][2] + m[1][1] * m[2][2] -
                   m[1][2] * m[1][2];
  const float c2 = m[0][0] + m[1][1] + m[2][2];
  if (std::fabs(c0) < std::numeric_limits<float>::epsilon()) {
    roots2(c2, c1, r);
    return;
  }
  const float s_inv3 = static_cast<float>(1.0 / 3.0);
  const float s_sqrt3 = std::sqrt(3.0f);
  const float c2_over_3 = c2 * s_inv3;
  float a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
  if (a_over_3 > 0.0f) a_over_3 = 0.0f;
  const float half_b = 0.5f * (c0 + c2_over_3 * (2.0f * c2_over_3 * c2_over_3 - c1));
  float q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
  if (q > 0.0f) q = 0.0f;
  const float rho = std::sqrt(-a_over_3);
  const float theta = std::atan2(std::sqrt(-q), half_b) * s_inv3;
  const float cos_theta = std::cos(theta);
  const float sin_theta = std::sin(theta);
  r[0] = c2_over_3 + 2.0f * rho * cos_theta;
  r[1] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
  r[2] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
  if (r[0] >= r[1]) std::swap(r[0], r[1]);
  if (r[1] >= r[2]) {
    std::swap(r[1], r[2]);
    if (r[0] >= r[1]) std::swap(r[0], r[1]);
  }
  if (r[0] <= 0.0f) roots2(c2, c1, r);
}

void smallest_eigenvector(const float cov[3][3], float* vec) {
  float scale = 0.0f;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) scale = std::max(scale, std::fabs(cov[i][j]));
  if (scale <= std::numeric_limits<float>::min()) scale = 1.0f;
  float m[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) m[i][j] = cov[i][j] / scale;
  float r[3];
  roots3(m, r);
  for (int i = 0; i < 3; ++i) m[i][i] -= r[0];
  auto cross = [](const float* a, const float* b, float* o) {
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
  };
  float v1[3], v2[3], v3[3];
  cross(m[0], m[1], v1);
  cross(m[0], m[2], v2);
  cross(m[1], m[2], v3);
  auto sq = [](const float* a) { return a[0] * a[0] + a[1] * a[1] + a[2] * a[2]; };
  const float l1 = sq(v1), l2 = sq(v2), l3 = sq(v3);
  const float* best = v3;
  float len = l3;
  if (l1 >= l2 && l1 >= l3) { best = v1; len = l1; }
  else if (l2 >= l1 && l2 >= l3) { best = v2; len = l2; }
  const float s = std::sqrt(len);
  for (int a = 0; a < 3; ++a) vec[a] = best[a] / s;
}
}  // namespace

/* Known-answer hook for the sampler: the i-th output (0-based) of mt19937 seeded with `seed`. */
uint32_t cmo_mt19937_at(uint32_t seed, int64_t i) {
  Mt19937 g(seed);
  uint32_t v = 0;
  for (int64_t k = 0; k <= i; ++k) v = g.next();
  return v;
}

/* Scores one externally given sample (three indices): coeff[4], returns the inlier count or -1 for a bad sample. */
int64_t cmo_plane_score(const float* xyzi, int64_t n, const int32_t* sample, double threshold, int32_t sum_order,
                        float* coeff) {
  const float *p0 = xyzi + 4 * static_cast<int64_t>(sample[0]), *p1 = xyzi + 4 * static_cast<int64_t>(sample[1]),
              *p2 = xyzi + 4 * static_cast<int64_t>(sample[2]);
  if (!plane_sample_good(p0, p1, p2)) return -1;
  plane_from_sample(p0, p1, p2, sum_order, coeff);
  int64_t cnt = 0;
  for (int64_t i = 0; i < n; ++i)
    if (plane_distance(coeff, xyzi + 4 * i, sum_order) < threshold) ++cnt;
  return cnt;
}

/* The whole segment() call. out_info: [0] found, [1] iterations, [2] draws taken from the sampler, [3] inlier count of
 * the best RANSAC model, [4..6] its sample. coeff_ransac / coeff_out: the RANSAC model and what segment() returns
 * (refined when optimize != 0). out_inliers [n]: the final inlier indices, ascending. Returns their number (0 when no
 * model was found). */
int64_t cmo_plane_ransac(const float* xyzi, int64_t n, double threshold, double probability, int32_t max_iterations,
                         int32_t optimize, uint32_t seed, int32_t sum_order, int32_t* out_info, float* coeff_ransac,
                         float* coeff_out, int32_t* out_inliers) {
  int32_t info[7] = {0, 0, 0, 0, -1, -1, -1};
  auto finish = [&](int64_t k) {
    if (out_info) std::memcpy(out_info, info, sizeof(info));
    return k;
  };
  if (n < 3) return finish(0);
  std::vector<int32_t> shuffled(static_cast<size_t>(n));
  for (int64_t i = 0; i < n; ++i) shuffled[i] = static_cast<int32_t>(i);
  Mt19937 rng(seed);
  int iterations = 0, draws = 0;
  int64_t best = -std::numeric_limits<int>::max();
  double k = 1.0;
  const double log_probability = std::log(1.0 - probability);
  const double one_over_indices = 1.0 / static_cast<double>(n);
  float best_c[4] = {0, 0, 0, 0};
  bool have = false;
  while (iterations < k) {
    int32_t sel[3];
    bool got = false;
    for (int check = 0; check < 1000 && !got; ++check) {
      for (int64_t i = 0; i < 3; ++i) {
        const int32_t r = static_cast<int32_t>(rng.next() >> 1);
        std::swap(shuffled[i], shuffled[i + static_cast<int64_t>(static_cast<uint64_t>(r) % static_cast<uint64_t>(n - i))]);
      }
      ++draws;
      sel[0] = shuffled[0]; sel[1] = shuffled[1]; sel[2] = shuffled[2];
      got = plane_sample_good(xyzi + 4 * static_cast<int64_t>(sel[0]), xyzi + 4 * static_cast<int64_t>(sel[1]),
                              xyzi + 4 * static_cast<int64_t>(sel[2]));
    }
    if (!got) break;
    float c[4];
    plane_from_sample(xyzi + 4 * static_cast<int64_t>(sel[0]), xyzi + 4 * static_cast<int64_t>(sel[1]),
                      xyzi + 4 * static_cast<int64_t>(sel[2]), sum_order, c);
    int64_t cnt = 0;
    for (int64_t i = 0; i < n; ++i)
      if (plane_distance(c, xyzi + 4 * i, sum_order) < threshold) ++cnt;
    if (cnt > best) {
      best = cnt;
      have = true;
      std::memcpy(best_c, c, sizeof(c));
      info[3] = static_cast<int32_t>(cnt);
      info[4] = sel[0]; info[5] = sel[1]; info[6] = sel[2];
      const double w = static_cast<double>(best) * one_over_indices;
      double p_no_outliers = 1.0 - std::pow(w, 3.0);
      p_no_outliers = std::max(std::numeric_limits<double>::epsilon(), p_no_outliers);
      p_no_outliers = std::min(1.0 - std::numeric_limits<double>::epsilon(), p_no_outliers);
      k = log_probability / std::log(p_no_outliers);
    }
    ++iterations;
    if (iterations > max_iterations) break;
  }
  info[1] = iterations;
  info[2] = draws;
  if (!have) return finish(0);
  info[0] = 1;
  if (coeff_ransac) std::memcpy(coeff_ransac, best_c, sizeof(best_c));
  std::vector<int32_t> inl;
  auto select = [&](const float* c) {
    inl.clear();
    for (int64_t i = 0; i < n; ++i)
      if (plane_distance(c, xyzi + 4 * i, sum_order) < threshold) inl.push_back(static_cast<int32_t>(i));
  };
  select(best_c);
  float fin_c[4];
  std::memcpy(fin_c, best_c, sizeof(fin_c));
  if (optimize) {
    if (inl.size() >= 4) {
      float acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
      for (int32_t i : inl) {
        const float* p = xyzi + 4 * static_cast<int64_t>(i);
        acc[0] += p[0] * p[0];
        acc[1] += p[0] * p[1];
        acc[2] += p[0] * p[2];
        acc[3] += p[1] * p[1];
        acc[4] += p[1] * p[2];
        acc[5] += p[2] * p[2];
        acc[6] += p[0];
        acc[7] += p[1];
        acc[8] += p[2];
      }
      const float cnt = static_cast<float>(inl.size());
      for (int a = 0; a < 9; ++a) acc[a] = acc[a] / cnt;
      float cov[3][3];
      cov[0][0] = acc[0] - acc[6] * acc[6];
      cov[0][1] = acc[1] - acc[6] * acc[7];
      cov[0][2] = acc[2] - acc[6] * acc[8];
      cov[1][1] = acc[3] - acc[7] * acc[7];
      cov[1][2] = acc[4] - acc[7] * acc[8];
      cov[2][2] = acc[5] - acc[8] * acc[8];
      cov[1][0] = cov[0][1]; cov[2][0] = cov[0][2]; cov[2][1] = cov[1][2];
      float v[3];
      smallest_eigenvector(cov, v);
      fin_c[0] = v[0]; fin_c[1] = v[1]; fin_c[2] = v[2];
      fin_c[3] = -1.0f * sum4(v[0] * acc[6], v[1] * acc[7], v[2] * acc[8], 0.0f * 1.0f, sum_order);
    }
    select(fin_c);
  }
  if (coeff_out) std::memcpy(coeff_out, fin_c, sizeof(fin_c));
  if (out_inliers) std::memcpy(out_inliers, inl.data(), inl.size() * sizeof(int32_t));
  return finish(static_cast<int64_t>(inl.size()));
}

const char* cmo_version(void) { return "cm_oracle 1 (PCL 1.8.1 restatement; parity unpinned)"; }

}  // extern "C"
