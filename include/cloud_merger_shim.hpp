// cloud_merger_shim.hpp -- header-only C++ host layer over the C ABI (cloud_merger_gpu.h) that re-creates the reference's
// own function surface for the merge hot path, so a maintainer can swap the PCL calls for the GPU path without touching
// the ROS node shell:
//
//   reference (pc_preprocessing_main.h:80-88, CloudFusionNode.h:59,145,276)      here (namespace cloud_merger)
//   pcl_ros::transformPointCloud(const Cloud&, Cloud&, const tf::Transform&)  ->  transformPointCloud(in, out, Transform)
//   void getROI(const Cloud::Ptr, Cloud::Ptr)                                 ->  getROI(in, out)
//   void getCloudPart(const Cloud::Ptr, Cloud::Ptr, float length, float dev)  ->  getCloudPart(in, out, length, deviation)
//   proceedX: getCloudPart x5 + the z windows of removeGround                 ->  getCloudPartsZSplit (one GPU pass)
//   void fusePointclouds(Cloud::Ptr no_ground, Cloud::Ptr ground)             ->  FusedFrame::fuse (+ operator+= kept)
//   void outlierRemoval(Cloud::Ptr)                                           ->  outlierRemoval(cloud)
//   proceedX after getROI: 5 x (getCloudPart + removeGround), appended          ->  proceedZones(ctx, roi, parts, no_ground, ground)
//   void removeGround(cloud, no_ground, ground, z_min, z_max, max_angle)      ->  removeGround(...) (z windows + RANSAC
//                                                                                 plane + ExtractIndices + outlierRemoval)
//   void voxelgrid(const Cloud::Ptr, Cloud::Ptr)                              ->  voxelgrid(in, out)
//   callbackX(const Cloud input) ... main loop fuse + voxelgrid               ->  FusedFrame::onCloud / fuseAndVoxel
//
// Cloud = pcl::PointCloud<pcl::PointXYZI> when PCL is present; otherwise the layout-compatible stand-ins below (PCL is
// not installed in the build image, so the tests use the stand-ins; the record layout -- 32 bytes, x y z at 0 4 8,
// pad 1.0f at 12, intensity at 16 -- is PCL's own, which makes every copy in and out a memcpy).
//
// Error behaviour mirrors the reference: the functions are void; on a GPU / capacity error they leave the output empty
// and report through last_error() (PCL itself only PCL_WARNs). No CPU fallback exists.
#ifndef CLOUD_MERGER_SHIM_HPP_
#define CLOUD_MERGER_SHIM_HPP_

#include <atomic>
#include <cstdint>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "cloud_merger_gpu.h"

#if defined(__has_include)
#if __has_include(<pcl/point_cloud.h>) && __has_include(<pcl/point_types.h>) && !defined(CM_SHIM_NO_PCL)
#include <pcl/point_cloud.h>
#include <pcl/point_types.h>
#define CM_SHIM_HAVE_PCL 1
#endif
#endif

// Optional adapters for the types either side of the path; each block compiles only where its header exists (ROS Melodic
// has all of them; the build image has none, so tests/cpp/mock/ carries minimal stand-ins with the same member names).
#if defined(__has_include)
#if __has_include(<sensor_msgs/PointCloud2.h>) && !defined(CM_SHIM_NO_ROS)
#include <sensor_msgs/PointCloud2.h>
#define CM_SHIM_HAVE_ROS_MSG 1
#endif
#if __has_include(<Eigen/Core>) && !defined(CM_SHIM_NO_EIGEN)
#include <Eigen/Core>
#define CM_SHIM_HAVE_EIGEN 1
#endif
#if __has_include(<tf/transform_datatypes.h>) && !defined(CM_SHIM_NO_ROS)
#include <tf/transform_datatypes.h>
#define CM_SHIM_HAVE_TF 1
#endif
#endif

namespace cloud_merger {

#ifdef CM_SHIM_HAVE_PCL
using PointXYZI = pcl::PointXYZI;
using Cloud = pcl::PointCloud<pcl::PointXYZI>;
inline uint64_t stamp_of(const Cloud& c) { return c.header.stamp; }
inline void set_stamp(Cloud& c, uint64_t s) { c.header.stamp = s; }
#else
// pcl::PointXYZI (point_types.hpp): PCL_ADD_POINT4D + intensity, 16-byte aligned, sizeof == 32.
struct alignas(16) PointXYZI {
  float x = 0.f, y = 0.f, z = 0.f, data3 = 1.f;
  float intensity = 0.f, data_c1 = 0.f, data_c2 = 0.f, data_c3 = 0.f;
};
static_assert(sizeof(PointXYZI) == 32, "PointXYZI must match pcl::PointXYZI");
// the members of pcl::PointCloud<PointT> the reference touches
template <typename PointT>
struct PointCloudT {
  struct Header {
    uint64_t stamp = 0;
    std::string frame_id;
  } header;
  std::vector<PointT> points;
  uint32_t width = 0, height = 0;
  bool is_dense = true;
  using Ptr = std::shared_ptr<PointCloudT<PointT>>;
  size_t size() const { return points.size(); }
  // pcl::PointCloud::operator+= (PCL 1.8.1): append, newest stamp, width = size, height = 1, is_dense = AND
  PointCloudT& operator+=(const PointCloudT& rhs) {
    if (rhs.header.stamp > header.stamp) header.stamp = rhs.header.stamp;
    points.insert(points.end(), rhs.points.begin(), rhs.points.end());
    width = static_cast<uint32_t>(points.size());
    height = 1;
    is_dense = rhs.is_dense && is_dense;
    return *this;
  }
};
using Cloud = PointCloudT<PointXYZI>;
inline uint64_t stamp_of(const Cloud& c) { return c.header.stamp; }
inline void set_stamp(Cloud& c, uint64_t s) { c.header.stamp = s; }
#endif

// tf::Transform as the reference builds it: tf::Transform(stf.getRotation(), stf.getOrigin()) (pc_preprocessing_main.cpp:320)
struct Transform {
  double q[4] = {0, 0, 0, 1};  // quaternion x y z w
  double origin[3] = {0, 0, 0};
};

// Parameter.h:27-35 (pcl_preprocessing) -- the reference's compile-time constants
struct Params {
  float voxel_size = 0.1f;
  int points_per_voxel = 2;
  float roi_width = 10.0f, roi_length = 75.0f, roi_mid = 15.0f, roi_z_min = -0.5f, roi_z_max = 3.0f;
  float radius = 0.15f;      // outlier removal: radius [m] and minimum number of neighbours (Parameter.h:23-24)
  float min_neighbor = 1;
  // RANSAC ground plane (Parameter.h:38-42); sum_order: the instruction set the PCL binary being replaced was built for
  int max_iterations = 1000;
  float distance_threshold = 0.3f;
  float prob = 0.99f;
  int sum_order = CM_SUM4_SSE2;
  // per-sensor zone tables (Parameter.h:45-81): zone lengths along x and the ground window |z| <= z_max_ground of each zone
  float vf_front_length = 30.0f, vf_mid_length = 15.0f, vf_mid_length2 = 11.0f, vf_veh_length = 8.0f, vf_rear_length = 11.0f;
  float vf_z_max_ground_front = 2.5f, vf_z_max_ground_mid2 = 2.0f, vf_z_max_ground_mid = 1.5f, vf_z_max_ground_veh = 0.3f,
        vf_z_max_ground_rear = 0.5f;
  float vr_front_length = 30.0f, vr_mid_length = 26.0f, vr_veh_length = 8.0f, vr_rear_length = 11.0f;
  float vr_z_max_ground_front = 2.0f, vr_z_max_ground_mid = 1.5f, vr_z_max_ground_veh = 0.3f, vr_z_max_ground_rear = 0.5f;
  float vt_front_length = 40.0f, vt_deviation_start_point = 20.0f, vt_z_max_ground_front = 1.0f;
  float l_front_length = 26.0f, l_mid_length = 10.0f, l_mid2_length = 10.0f, l_rear_length = 10.0f, l_deviation_mid_point = 4.0f;
  float l_z_max_ground_front = 1.5f, l_z_max_ground_mid2 = 1.2f, l_z_max_ground_mid = 0.8f, l_z_max_ground_rear = 0.5f;
};

// my_cloud_fusion/src/Parameter.h:15-110 -- that package's constants are `double` (narrowed to float where PCL takes them)
struct FusionParams {
  double radius = 0.1, min_neighbor = 1;
  double x_transverse = 20.0, y_transverse = 25.0, x_longitudinal = 30.0, y_longitudinal = 10.0, z_min = -0.5, z_max = 3.0;
  double lane_width = 10.0;
  int points_per_voxel = 2;
  double voxel_size = 0.1;
  // zone lengths and ground windows per sensor group: [0] front Velodynes, [1] rear Velodynes, [2] top Velodyne, [3] Livox
  // (Parameter.h:37-105; proceed_pointcloud picks the group by cloud index, CloudFusionNode.h:346-413)
  struct Group {
    double front_length, mid_length, rear_length;
    double z_min_ground_front, z_max_ground_front, z_min_ground_mid, z_max_ground_mid, z_min_ground_rear, z_max_ground_rear;
  };
  Group group[4] = {{15.0, 10.0, 10.0, -0.5, 0.5, -0.2, 0.2, -0.5, 0.5},
                    {10.0, 10.0, 15.0, -0.5, 0.5, -0.2, 0.2, -0.5, 0.5},
                    {40.0, 40.0, 0.0, -1.5, 1.5, -0.5, 0.5, -0.5, 0.5},
                    {10.0, 20.0, 0.0, -0.5, 0.5, -0.5, 0.5, -0.5, 0.5}};
};

inline cm_layout_t pcl_layout(bool is_dense) {
  cm_layout_t l;
  l.point_step = 32; l.off_x = 0; l.off_y = 4; l.off_z = 8; l.off_intensity = 16; l.is_dense = is_dense ? 1 : 0;
  return l;
}

// One GPU context shared by the drop-in functions. Capacity = largest single cloud / fused frame it will be handed.
class Context {
 public:
  explicit Context(int64_t max_points_per_cloud = 1 << 20, int max_sensors = 6, int device = 0, Params p = Params())
      : params_(p), max_points_(max_points_per_cloud), max_sensors_(max_sensors) {
    cm_config_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.device = device;
    cfg.max_sensors = max_sensors;
    cfg.max_points_per_sensor = max_points_per_cloud;
    cfg.max_point_step = 32;
    cfg.frames_in_flight = 2;
    cfg.max_batch_points = max_points_per_cloud * max_sensors;
    cfg.max_batch_frames = CM_MAX_ZONES;  // several zone clouds per radius_outlier_multi call
    cfg.out_point_step = 32;  // pcl::PointXYZI records straight out of the kernels
    rc_ = cm_create(&cfg, &h_);
    if (rc_ != CM_OK) { h_ = nullptr; err_ = cm_strerror(rc_); }
  }
  ~Context() {
    if (h_) {
      if (dev_in_) cm_dev_free(h_, dev_in_);
      cm_destroy(h_);
    }
  }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;

  bool ok() const { return h_ != nullptr; }
  cm_handle_t handle() const { return h_; }
  const Params& params() const { return params_; }
  const std::string& last_error() const { return err_; }
  int last_status() const { return rc_; }

  // transform + crop of ONE host cloud (stage entry cm_dev_transform_crop); out keeps input order.
  bool transform_crop(const Cloud& in, Cloud& out, const float* m16_row_major, int n_pass, const cm_pass_t* passes) {
    if (!check(h_ ? CM_OK : CM_E_NO_DEVICE)) return clear(out);
    const int64_t n = static_cast<int64_t>(in.points.size());
    if (n > max_points_) { rc_ = CM_E_CAPACITY; err_ = "cloud larger than the context capacity"; return clear(out); }
    if (!stage_in(in.points.data(), n)) return clear(out);
    if (!check(cm_set_extrinsic(h_, 0, m16_row_major, 0)) || !check(cm_set_crop(h_, n_pass, passes))) return clear(out);
    cm_segment_t seg;
    seg.data = dev_in_; seg.n_points = n; seg.layout = pcl_layout(in.is_dense); seg.sensor = 0; seg.frame = 0;
    if (!check(cm_dev_transform_crop(h_, &seg, 1, nullptr))) return clear(out);
    cm_stats_t st;
    cm_device_out_t o;
    if (!check(cm_get_stats(h_, &st)) || !check(cm_get_device_out(h_, &o))) return clear(out);
    const size_t m = static_cast<size_t>(st.survivors);
    tmp_.resize(m * 4);
    if (m && !check(cm_memcpy_d2h(h_, tmp_.data(), o.survivor_xyzi, m * 16, nullptr))) return clear(out);
    out.points.resize(m);
    for (size_t i = 0; i < m; ++i) {
      PointXYZI& p = out.points[i];
      p = PointXYZI();
      p.x = tmp_[i * 4 + 0]; p.y = tmp_[i * 4 + 1]; p.z = tmp_[i * 4 + 2]; p.intensity = tmp_[i * 4 + 3];
    }
    finish(out, in, n_pass > 0 ? true : in.is_dense);
    return true;
  }

  // VoxelGrid of ONE host cloud (stage entry cm_dev_voxelgrid).
  bool voxelgrid(const Cloud& in, Cloud& out) {
    if (!check(h_ ? CM_OK : CM_E_NO_DEVICE)) return clear(out);
    const int64_t n = static_cast<int64_t>(in.points.size());
    if (n > max_points_ * max_sensors_) { rc_ = CM_E_CAPACITY; err_ = "cloud larger than the context capacity"; return clear(out); }
    // the voxel stage reads packed xyzi
    tmp_.resize(static_cast<size_t>(n) * 4);
    for (int64_t i = 0; i < n; ++i) {
      const PointXYZI& p = in.points[static_cast<size_t>(i)];
      tmp_[i * 4 + 0] = p.x; tmp_[i * 4 + 1] = p.y; tmp_[i * 4 + 2] = p.z; tmp_[i * 4 + 3] = p.intensity;
    }
    if (!stage_in(tmp_.data(), n, 16)) return clear(out);
    const float leaf[3] = {params_.voxel_size, params_.voxel_size, params_.voxel_size};
    if (!check(cm_set_voxel(h_, leaf, params_.points_per_voxel, 1))) return clear(out);
    if (!check(cm_dev_voxelgrid(h_, static_cast<const float*>(dev_in_), n, in.is_dense ? 1 : 0, nullptr))) return clear(out);
    cm_stats_t st;
    cm_device_out_t o;
    if (!check(cm_get_stats(h_, &st)) || !check(cm_get_device_out(h_, &o))) return clear(out);
    if (st.pcl_overflow) {  // PCL 1.8.1: "Leaf size is too small for the input dataset" -> output = input
      out = in;
      return true;
    }
    const size_t v = static_cast<size_t>(st.voxels_out);
    out.points.resize(v);
    if (v && !check(cm_memcpy_d2h(h_, out.points.data(), o.voxel_xyzi, v * 32, nullptr))) return clear(out);
    finish(out, in, true);
    return true;
  }

  // Radius outlier removal of several host clouds in one pass (cm_radius_outlier_multi; at most CM_MAX_ZONES clouds):
  // every cloud is filtered on its own (no neighbours across clouds); out[k] keeps the order of in[k].
  bool radius_outlier_multi(const std::vector<const Cloud*>& in, std::vector<Cloud>& out, double radius, int min_neighbors) {
    return filter_multi(in, out, [&](const int64_t* begin, int k, int64_t n, int64_t* ob) {
      return cm_radius_outlier_multi(h_, tmp_.data(), begin, k, radius, min_neighbors, 0, zone_xyzi_.data(), nullptr, n, ob);
    });
  }
  // one cloud
  bool radius_outlier(const Cloud& in, Cloud& out, double radius, int min_neighbors) {
    std::vector<Cloud> res;
    if (!radius_outlier_multi({&in}, res, radius, min_neighbors)) return clear(out);
    out = res[0];
    return true;
  }

  // Statistical outlier removal of several host clouds in one pass (cm_statistical_outlier_multi; at most CM_MAX_ZONES
  // clouds): pcl::StatisticalOutlierRemoval with setMeanK(mean_k), setStddevMulThresh(std_mul), setNegative(negative) on
  // every cloud on its own; out[k] keeps the order of in[k]. sqrt_mode: CM_SOR_SQRT_FLOAT / CM_SOR_SQRT_DOUBLE, the
  // reading of the unqualified sqrt in PCL's loop that the build being replaced makes.
  bool statistical_outlier_multi(const std::vector<const Cloud*>& in, std::vector<Cloud>& out, int mean_k, double std_mul,
                                 bool negative = false, int sqrt_mode = CM_SOR_SQRT_FLOAT) {
    cm_sor_cfg_t cfg{};
    cfg.mean_k = mean_k; cfg.negative = negative ? 1 : 0; cfg.sqrt_mode = sqrt_mode; cfg.std_mul = std_mul;
    return filter_multi(in, out, [&](const int64_t* begin, int k, int64_t n, int64_t* ob) {
      return cm_statistical_outlier_multi(h_, tmp_.data(), begin, k, &cfg, zone_xyzi_.data(), nullptr, n, ob);
    });
  }
  bool statistical_outlier(const Cloud& in, Cloud& out, int mean_k, double std_mul, bool negative = false,
                           int sqrt_mode = CM_SOR_SQRT_FLOAT) {
    std::vector<Cloud> res;
    if (!statistical_outlier_multi({&in}, res, mean_k, std_mul, negative, sqrt_mode)) return clear(out);
    out = res[0];
    return true;
  }

  // RANSAC ground plane of several host clouds in one pass (cm_plane_ransac_multi; at most CM_MAX_ZONES / 2 clouds): per
  // cloud pcl::SACSegmentation (SACMODEL_PLANE, SAC_RANSAC, optimize on) + the two pcl::ExtractIndices passes;
  // ground[k] = the inliers of in[k], no_ground[k] = its other points, both in input order.
  bool plane_ransac_multi(const std::vector<const Cloud*>& in, std::vector<Cloud>& ground, std::vector<Cloud>& no_ground,
                          std::vector<cm_plane_t>* models = nullptr) {
    const size_t k = in.size();
    ground.assign(k, Cloud()); no_ground.assign(k, Cloud());
    if (!check(h_ ? CM_OK : CM_E_NO_DEVICE)) return false;
    std::vector<int64_t> begin(k + 1, 0);
    for (size_t c = 0; c < k; ++c) begin[c + 1] = begin[c] + static_cast<int64_t>(in[c]->points.size());
    const int64_t n = begin[k];
    if (n > max_points_ * max_sensors_) { rc_ = CM_E_CAPACITY; err_ = "clouds larger than the context capacity"; return false; }
    tmp_.resize(static_cast<size_t>(n) * 4 + 4);
    for (size_t c = 0; c < k; ++c)
      for (size_t i = 0; i < in[c]->points.size(); ++i) {
        const PointXYZI& p = in[c]->points[i];
        float* o = &tmp_[(static_cast<size_t>(begin[c]) + i) * 4];
        o[0] = p.x; o[1] = p.y; o[2] = p.z; o[3] = p.intensity;
      }
    cm_plane_cfg_t cfg;
    cfg.distance_threshold = static_cast<double>(params_.distance_threshold);
    cfg.probability = static_cast<double>(params_.prob);
    cfg.max_iterations = params_.max_iterations;
    cfg.optimize = 1;
    cfg.seed = 12345u;
    cfg.sum_order = params_.sum_order;
    std::vector<cm_plane_t> pl(k);
    std::vector<int64_t> ob(2 * k + 1, 0);
    zone_xyzi_.resize(static_cast<size_t>(n) * 4 + 4);
    if (!check(cm_plane_ransac_multi(h_, tmp_.data(), begin.data(), static_cast<int>(k), &cfg, pl.data(), zone_xyzi_.data(),
                                     nullptr, n, ob.data())))
      return false;
    if (models) *models = pl;
    for (size_t z = 0; z < 2 * k; ++z) {
      Cloud& c = (z & 1) ? no_ground[z / 2] : ground[z / 2];
      const size_t b = static_cast<size_t>(ob[z]), e = static_cast<size_t>(ob[z + 1]);
      c.points.resize(e - b);
      for (size_t i = b; i < e; ++i) {
        PointXYZI& p = c.points[i - b];
        p = PointXYZI();
        p.x = zone_xyzi_[i * 4 + 0]; p.y = zone_xyzi_[i * 4 + 1]; p.z = zone_xyzi_[i * 4 + 2]; p.intensity = zone_xyzi_[i * 4 + 3];
      }
      finish(c, *in[z / 2], in[z / 2]->is_dense);
    }
    return true;
  }
  // one cloud
  bool plane_ransac(const Cloud& in, Cloud& ground, Cloud& no_ground, cm_plane_t* model = nullptr) {
    std::vector<Cloud> g, r;
    std::vector<cm_plane_t> m;
    const bool ok = plane_ransac_multi({&in}, g, r, &m);
    if (ok) { ground = g[0]; no_ground = r[0]; if (model) *model = m[0]; }
    else { clear(ground); clear(no_ground); }
    return ok;
  }

  // The body of a proceedX after getROI in ONE library call (cm_proceed_zones): every x / z window, the plane search of every
  // ground window, the outlier removal of what is not ground and the appends stay on the device in between.
  bool proceed(const Cloud& roi, const cm_proceed_cfg_t& cfg, Cloud& no_ground, Cloud& ground, std::vector<cm_plane_t>* models = nullptr) {
    if (!check(h_ ? CM_OK : CM_E_NO_DEVICE)) { clear(no_ground); return clear(ground); }
    const int64_t n = static_cast<int64_t>(roi.points.size());
    tmp_.resize(static_cast<size_t>(n) * 4 + 4);
    for (int64_t i = 0; i < n; ++i) {
      const PointXYZI& p = roi.points[static_cast<size_t>(i)];
      tmp_[i * 4 + 0] = p.x; tmp_[i * 4 + 1] = p.y; tmp_[i * 4 + 2] = p.z; tmp_[i * 4 + 3] = p.intensity;
    }
    const int64_t cap = 2 * n + 16;
    zone_xyzi_.resize(static_cast<size_t>(cap) * 4);
    std::vector<float> g(static_cast<size_t>(cap) * 4);
    int64_t n_ng = 0, n_g = 0;
    cm_plane_t pl[CM_MAX_PROCEED_PARTS];
    if (!check(cm_proceed_zones(h_, tmp_.data(), n, &cfg, zone_xyzi_.data(), cap, &n_ng, g.data(), cap, &n_g, pl))) {
      clear(no_ground);
      return clear(ground);
    }
    auto fill = [&](Cloud& c, const float* src, int64_t k) {
      c.points.resize(static_cast<size_t>(k));
      for (int64_t i = 0; i < k; ++i) {
        PointXYZI& p = c.points[static_cast<size_t>(i)];
        p = PointXYZI();
        p.x = src[i * 4 + 0]; p.y = src[i * 4 + 1]; p.z = src[i * 4 + 2]; p.intensity = src[i * 4 + 3];
      }
      finish(c, roi, true);
    };
    fill(no_ground, zone_xyzi_.data(), n_ng);
    fill(ground, g.data(), n_g);
    if (models) {
      models->clear();
      for (int k = 0, c = 0; k < cfg.n_parts; ++k)
        if (cfg.part[k].ground_removal) models->push_back(pl[c++]);
    }
    return true;
  }

  // Zone slicing of ONE host cloud (cm_zone_split): one ordered output cloud per PassThrough chain, one GPU pass.
  bool zone_split(const Cloud& in, const std::vector<cm_zone_t>& zones, std::vector<Cloud>& out) {
    out.assign(zones.size(), Cloud());
    if (!check(h_ ? CM_OK : CM_E_NO_DEVICE)) return false;
    const int64_t n = static_cast<int64_t>(in.points.size());
    tmp_.resize(static_cast<size_t>(n) * 4);
    for (int64_t i = 0; i < n; ++i) {
      const PointXYZI& p = in.points[static_cast<size_t>(i)];
      tmp_[i * 4 + 0] = p.x; tmp_[i * 4 + 1] = p.y; tmp_[i * 4 + 2] = p.z; tmp_[i * 4 + 3] = p.intensity;
    }
    if (!check(cm_set_zones(h_, static_cast<int>(zones.size()), zones.data()))) return false;
    int64_t begin[CM_MAX_ZONES + 1] = {0};
    int64_t cap = 2 * n + 16;
    zone_xyzi_.resize(static_cast<size_t>(cap) * 4);
    int rc = cm_zone_split(h_, tmp_.data(), n, zone_xyzi_.data(), nullptr, cap, begin);
    if (rc == CM_E_CAPACITY && begin[zones.size()] > cap) {  // heavily overlapping zones: the needed size came back
      cap = begin[zones.size()];
      zone_xyzi_.resize(static_cast<size_t>(cap) * 4);
      rc = cm_zone_split(h_, tmp_.data(), n, zone_xyzi_.data(), nullptr, cap, begin);
    }
    if (!check(rc)) return false;
    for (size_t z = 0; z < zones.size(); ++z) {
      Cloud& c = out[z];
      const size_t b = static_cast<size_t>(begin[z]), e = static_cast<size_t>(begin[z + 1]);
      c.points.resize(e - b);
      for (size_t i = b; i < e; ++i) {
        PointXYZI& p = c.points[i - b];
        p = PointXYZI();
        p.x = zone_xyzi_[i * 4 + 0]; p.y = zone_xyzi_[i * 4 + 1]; p.z = zone_xyzi_[i * 4 + 2]; p.intensity = zone_xyzi_[i * 4 + 3];
      }
      finish(c, in, zones[z].n_pass > 0 ? true : in.is_dense);
    }
    return true;
  }

 private:
  // Packs the clouds into tmp_ (xyzi), runs a multi-cloud filter of the C ABI that writes the survivors of cloud c to
  // zone_xyzi_[ob[c] .. ob[c+1]) and unpacks them into out[c] (header and layout of in[c]).
  template <typename Run>
  bool filter_multi(const std::vector<const Cloud*>& in, std::vector<Cloud>& out, Run run) {
    const size_t k = in.size();
    out.assign(k, Cloud());
    if (!check(h_ ? CM_OK : CM_E_NO_DEVICE)) return false;
    std::vector<int64_t> begin(k + 1, 0);
    for (size_t c = 0; c < k; ++c) begin[c + 1] = begin[c] + static_cast<int64_t>(in[c]->points.size());
    const int64_t n = begin[k];
    if (n > max_points_ * max_sensors_) { rc_ = CM_E_CAPACITY; err_ = "clouds larger than the context capacity"; return false; }
    tmp_.resize(static_cast<size_t>(n) * 4 + 4);
    for (size_t c = 0; c < k; ++c)
      for (size_t i = 0; i < in[c]->points.size(); ++i) {
        const PointXYZI& p = in[c]->points[i];
        float* o = &tmp_[(static_cast<size_t>(begin[c]) + i) * 4];
        o[0] = p.x; o[1] = p.y; o[2] = p.z; o[3] = p.intensity;
      }
    zone_xyzi_.resize(static_cast<size_t>(n) * 4 + 4);
    std::vector<int64_t> ob(k + 1, 0);
    if (!check(run(begin.data(), static_cast<int>(k), n, ob.data()))) return false;
    for (size_t c = 0; c < k; ++c) {
      Cloud& res = out[c];
      const size_t b = static_cast<size_t>(ob[c]), e = static_cast<size_t>(ob[c + 1]);
      res.points.resize(e - b);
      for (size_t i = b; i < e; ++i) {
        PointXYZI& p = res.points[i - b];
        p = PointXYZI();
        p.x = zone_xyzi_[i * 4 + 0]; p.y = zone_xyzi_[i * 4 + 1]; p.z = zone_xyzi_[i * 4 + 2]; p.intensity = zone_xyzi_[i * 4 + 3];
      }
      finish(res, *in[c], true);
    }
    return true;
  }

  bool check(int rc) {
    rc_ = rc;
    if (rc != CM_OK) err_ = std::string(cm_strerror(rc)) + ": " + (h_ ? cm_last_error(h_) : "");
    return rc == CM_OK;
  }
  static bool clear(Cloud& out) {
    out.points.clear(); out.width = 0; out.height = 1;
    return false;
  }
  static void finish(Cloud& out, const Cloud& in, bool dense) {
    out.width = static_cast<uint32_t>(out.points.size());
    out.height = 1;
    out.is_dense = dense;
    out.header = in.header;
  }
  bool stage_in(const void* host, int64_t n, int step = 32) {
    const size_t need = static_cast<size_t>(max_points_) * max_sensors_ * 32 + 64;
    if (!dev_in_ && !check(cm_dev_alloc(h_, &dev_in_, need))) return false;
    if (n == 0) return true;
    return check(cm_memcpy_h2d(h_, dev_in_, host, static_cast<size_t>(n) * step, nullptr));
  }

  Params params_;
  int64_t max_points_;
  int max_sensors_;
  cm_handle_t h_ = nullptr;
  void* dev_in_ = nullptr;
  std::vector<float> tmp_, zone_xyzi_;
  std::string err_;
  int rc_ = CM_OK;
};

inline void matrix_from_transform(const Transform& t, float* m16) {
  // pcl_ros::transformPointCloud: Eigen::Quaternionf(q.w, q.x, q.y, q.z), Vector3f(origin), Eigen 3.3 toRotationMatrix
  const float x = static_cast<float>(t.q[0]), y = static_cast<float>(t.q[1]), z = static_cast<float>(t.q[2]),
              w = static_cast<float>(t.q[3]);
  const float tx = 2.0f * x, ty = 2.0f * y, tz = 2.0f * z;
  const float twx = tx * w, twy = ty * w, twz = tz * w, txx = tx * x, txy = ty * x, txz = tz * x;
  const float tyy = ty * y, tyz = tz * y, tzz = tz * z;
  const float m[16] = {1.0f - (tyy + tzz), txy - twz, txz + twy, static_cast<float>(t.origin[0]),
                       txy + twz, 1.0f - (txx + tzz), tyz - twx, static_cast<float>(t.origin[1]),
                       txz - twy, tyz + twx, 1.0f - (txx + tyy), static_cast<float>(t.origin[2]),
                       0.f, 0.f, 0.f, 1.f};
  std::memcpy(m16, m, sizeof(m));
}

// ---- adapters for the types either side of the path -----------------------------------------------------------------------
#ifdef CM_SHIM_HAVE_EIGEN
// Eigen::Matrix4f is column-major (Matrix4f::data() order): the extrinsic goes in as it is stored.
inline int setExtrinsic(cm_handle_t h, int sensor, const Eigen::Matrix4f& m) { return cm_set_extrinsic(h, sensor, m.data(), 1); }
#endif
#ifdef CM_SHIM_HAVE_TF
// tf::Transform(stf.getRotation(), stf.getOrigin()) as the callbacks build it (pc_preprocessing_main.cpp:320)
inline Transform fromTf(const tf::Transform& t) {
  Transform r;
  const tf::Quaternion q = t.getRotation();
  r.q[0] = q.x(); r.q[1] = q.y(); r.q[2] = q.z(); r.q[3] = q.w();
  r.origin[0] = t.getOrigin().x(); r.origin[1] = t.getOrigin().y(); r.origin[2] = t.getOrigin().z();
  return r;
}
#endif
#ifdef CM_SHIM_HAVE_ROS_MSG
// sensor_msgs::PointCloud2 -> cm_layout_t: the field lookup the pcl_ros subscriber does (pc_preprocessing_main.cpp:520-525);
// msg.data can then be handed to cm_submit_cloud as it arrived (no deserialisation into pcl::PointXYZI, no by-value copy).
inline int layoutFromMsg(const sensor_msgs::PointCloud2& msg, cm_layout_t* out) {
  std::vector<cm_pc2_field_t> f(msg.fields.size());
  for (size_t i = 0; i < msg.fields.size(); ++i) {
    f[i].name = msg.fields[i].name.c_str(); f[i].offset = msg.fields[i].offset;
    f[i].datatype = msg.fields[i].datatype; f[i].count = msg.fields[i].count;
  }
  return cm_layout_from_pointcloud2(f.data(), static_cast<int>(f.size()), msg.point_step, msg.is_bigendian ? 1 : 0,
                                    msg.is_dense ? 1 : 0, out);
}
// What pcl::toROSMsg(cloud, msg) does for a cloud of `n` records as the kernels write them (pc_preprocessing_main.cpp:199-220):
// header fields + one memcpy of the records. out_point_step 32 = pcl::PointXYZI records, 16 = packed xyzi.
inline bool fillMsg(sensor_msgs::PointCloud2& msg, const void* records, int64_t n, int out_point_step = 32) {
  cm_pc2_desc_t d;
  if (cm_pointcloud2_describe(out_point_step, n, &d) != CM_OK) return false;
  msg.height = d.height; msg.width = d.width; msg.point_step = d.point_step; msg.row_step = d.row_step;
  msg.is_bigendian = d.is_bigendian != 0; msg.is_dense = d.is_dense != 0;
  msg.fields.resize(static_cast<size_t>(d.n_fields));
  for (int k = 0; k < d.n_fields; ++k) {
    msg.fields[static_cast<size_t>(k)].name = d.fields[k].name; msg.fields[static_cast<size_t>(k)].offset = d.fields[k].offset;
    msg.fields[static_cast<size_t>(k)].datatype = d.fields[k].datatype; msg.fields[static_cast<size_t>(k)].count = d.fields[k].count;
  }
  msg.data.resize(static_cast<size_t>(d.row_step));
  if (d.row_step) std::memcpy(msg.data.data(), records, d.row_step);
  return true;
}
inline bool toROSMsg(const Cloud& cloud, sensor_msgs::PointCloud2& msg) {
  if (!fillMsg(msg, cloud.points.data(), static_cast<int64_t>(cloud.points.size()), 32)) return false;
  msg.is_dense = cloud.is_dense;
  return true;
}
#endif

// ---- the reference's functions, same names and argument meaning -------------------------------------------------------

// pcl_ros::transformPointCloud(input, *cloud_ptr, transform) -- pc_preprocessing_main.cpp:322
inline void transformPointCloud(Context& ctx, const Cloud& in, Cloud& out, const Transform& tf) {
  float m[16];
  matrix_from_transform(tf, m);
  ctx.transform_crop(in, out, m, 0, nullptr);
}

// void getROI(const Cloud::Ptr cloud_ptr, Cloud::Ptr cloud_ROI_ptr) -- pc_preprocessing_main.cpp:20-40
inline void getROI(Context& ctx, const Cloud::Ptr& cloud_ptr, const Cloud::Ptr& cloud_ROI_ptr) {
  const Params& p = ctx.params();
  const cm_pass_t passes[3] = {{2, p.roi_z_min, p.roi_z_max, 0},
                               {1, -p.roi_width / 2, p.roi_width / 2, 0},
                               {0, -p.roi_mid, p.roi_length - p.roi_mid, 0}};
  const float eye[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  Cloud tmp;
  ctx.transform_crop(*cloud_ptr, tmp, eye, 3, passes);
  *cloud_ROI_ptr = tmp;
}

// void getCloudPart(const Cloud::Ptr, Cloud::Ptr, const float length, const float deviation) -- :49-59
inline void getCloudPart(Context& ctx, const Cloud::Ptr& cloud_ptr, const Cloud::Ptr& cloud_part_ptr, const float length,
                         const float deviation) {
  const cm_pass_t pass = {0, deviation, deviation + length, 0};
  const float eye[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  Cloud tmp;
  ctx.transform_crop(*cloud_ptr, tmp, eye, 1, &pass);
  *cloud_part_ptr = tmp;
}

// The zone loop of proceedFront / proceedRear / proceedTop / proceedLivox (:228-312): for every part
//   getCloudPart(cloud_ROI_ptr, part, length, deviation);                                      -- x in [dev, dev + length]
//   removeGround(part, ...) { zpass [z_min_ground, z_max_ground]  -> ground_part_ptr;          -- :80-92, the input of RANSAC
//                             zpass2 [z_max_ground + 0.01, roi_z_max] -> no_ground_part_ptr }  -- appended after RANSAC
// i.e. 3 PassThrough runs + copies per part on the CPU; here all parts and both z windows come out of ONE GPU pass.
// z_min_ground is -z_max_ground at every call site of the reference. `z_max_ground + 0.01` is a double sum narrowed to
// float by setFilterLimits(const float&, const float&), exactly as in the reference.
struct ZonePart {
  float length, deviation, z_max_ground;
};
inline void getCloudPartsZSplit(Context& ctx, const Cloud::Ptr& cloud_ROI_ptr, const std::vector<ZonePart>& parts,
                                const float roi_z_max, std::vector<Cloud::Ptr>& ground_part_ptrs,
                                std::vector<Cloud::Ptr>& no_ground_part_ptrs) {
  std::vector<cm_zone_t> zones(parts.size() * 2);
  for (size_t k = 0; k < parts.size(); ++k) {
    const ZonePart& pt = parts[k];
    const cm_pass_t x = {0, pt.deviation, pt.deviation + pt.length, 0};
    const float z_lo2 = static_cast<float>(pt.z_max_ground + 0.01);
    zones[2 * k].n_pass = 2; zones[2 * k].pass[0] = x; zones[2 * k].pass[1] = cm_pass_t{2, -pt.z_max_ground, pt.z_max_ground, 0};
    zones[2 * k + 1].n_pass = 2; zones[2 * k + 1].pass[0] = x; zones[2 * k + 1].pass[1] = cm_pass_t{2, z_lo2, roi_z_max, 0};
  }
  std::vector<Cloud> out;
  ctx.zone_split(*cloud_ROI_ptr, zones, out);
  ground_part_ptrs.clear(); no_ground_part_ptrs.clear();
  for (size_t k = 0; k < parts.size(); ++k) {
    ground_part_ptrs.push_back(Cloud::Ptr(new Cloud(out[2 * k])));
    no_ground_part_ptrs.push_back(Cloud::Ptr(new Cloud(out[2 * k + 1])));
  }
}

// void outlierRemoval(Cloud::Ptr cloud_ptr) -- :184-192: pcl::RadiusOutlierRemoval, radius / min_neighbor of Parameter.h:23-24,
// filtering the cloud in place.
inline void outlierRemoval(Context& ctx, const Cloud::Ptr& cloud_ptr) {
  Cloud tmp;
  ctx.radius_outlier(*cloud_ptr, tmp, static_cast<double>(ctx.params().radius), static_cast<int>(ctx.params().min_neighbor));
  *cloud_ptr = tmp;
}

// pcl::StatisticalOutlierRemoval<PointXYZI> (setMeanK, setStddevMulThresh) filtering the cloud in place, next to
// outlierRemoval for a node that replaces its radius filter by PCL's other standard one.
inline void statisticalOutlierRemoval(Context& ctx, const Cloud::Ptr& cloud_ptr, int mean_k, double std_mul) {
  Cloud tmp;
  ctx.statistical_outlier(*cloud_ptr, tmp, mean_k, std_mul);
  *cloud_ptr = tmp;
}

// void removeGround(cloud, no_ground, ground, z_min_ground, z_max_ground, max_angle) -- :71-122, the whole function: the two
// z windows (one zone-slicing pass), the RANSAC plane on the lower one + ExtractIndices, outlierRemoval of what is not
// ground, and the points above the window appended. max_angle is accepted and unused, as in the reference (SACMODEL_PLANE
// ignores setAxis / setEpsAngle).
inline void removeGround(Context& ctx, const Cloud::Ptr& cloud_ptr, const Cloud::Ptr& no_ground_cloud_ptr,
                         const Cloud::Ptr& ground_cloud_ptr, const float z_min_ground, const float z_max_ground,
                         const float /*max_angle*/) {
  std::vector<cm_zone_t> zones(2);
  zones[0].n_pass = 1; zones[0].pass[0] = cm_pass_t{2, z_min_ground, z_max_ground, 0};
  zones[1].n_pass = 1; zones[1].pass[0] = cm_pass_t{2, static_cast<float>(z_max_ground + 0.01), ctx.params().roi_z_max, 0};
  std::vector<Cloud> parts;
  ctx.zone_split(*cloud_ptr, zones, parts);
  Cloud ground, no_ground;
  ctx.plane_ransac(parts[0], ground, no_ground);
  *ground_cloud_ptr = ground;
  *no_ground_cloud_ptr = no_ground;
  outlierRemoval(ctx, no_ground_cloud_ptr);
  *no_ground_cloud_ptr += parts[1];
}

// proceedFront / proceedRear / proceedTop / proceedLivox after getROI -- :228-312, :428-446, :474-497: per zone getCloudPart +
// removeGround, results appended zone after zone, `plain` x windows appended to the no-ground cloud unchanged. ONE library
// call (cm_proceed_zones): one zone-slicing pass for all x and z windows, one multi-cloud RANSAC pass for all ground windows,
// one multi-cloud outlierRemoval pass for what is not ground, the appends -- device-resident in between.
inline cm_proceed_cfg_t proceedConfig(const Params& p, const std::vector<ZonePart>& parts, const std::vector<ZonePart>& plain) {
  cm_proceed_cfg_t cfg;
  std::memset(&cfg, 0, sizeof(cfg));
  for (const ZonePart& pt : parts) {
    if (cfg.n_parts >= CM_MAX_PROCEED_PARTS) break;
    cfg.part[cfg.n_parts++] = cm_proceed_part_t{pt.length, pt.deviation, pt.z_max_ground, 1};
  }
  for (const ZonePart& pt : plain) {
    if (cfg.n_parts >= CM_MAX_PROCEED_PARTS) break;
    cfg.part[cfg.n_parts++] = cm_proceed_part_t{pt.length, pt.deviation, 0.0f, 0};
  }
  cfg.roi_z_max = p.roi_z_max;
  cfg.radius = static_cast<double>(p.radius);
  cfg.min_neighbors = static_cast<int>(p.min_neighbor);
  cfg.plane.distance_threshold = static_cast<double>(p.distance_threshold);
  cfg.plane.probability = static_cast<double>(p.prob);
  cfg.plane.max_iterations = p.max_iterations;
  cfg.plane.optimize = 1;
  cfg.plane.seed = 12345u;
  cfg.plane.sum_order = p.sum_order;
  return cfg;
}
inline void proceedZones(Context& ctx, const Cloud::Ptr& cloud_ROI_ptr, const std::vector<ZonePart>& parts,
                         const Cloud::Ptr& no_ground_ptr, const Cloud::Ptr& ground_ptr,
                         const std::vector<ZonePart>& plain = std::vector<ZonePart>()) {
  const cm_proceed_cfg_t cfg = proceedConfig(ctx.params(), parts, plain);
  Cloud ng, g;
  ctx.proceed(*cloud_ROI_ptr, cfg, ng, g);
  *no_ground_ptr = ng;
  *ground_ptr = g;
}

// ---- the zone tables of the four sensor groups (pc_preprocessing_main.cpp:228-312, :428-446, :474-497; Parameter.h:45-81) ----
// Deviations are the reference's own float expressions, summed left to right. `plain` parts are x windows that go to the
// no-ground cloud without ground removal (callbackTopMiddle's near range, :444-446).
struct ProceedTable {
  std::vector<ZonePart> parts;
  std::vector<ZonePart> plain;  // length, deviation; z_max_ground unused
};
inline ProceedTable frontTable(const Params& p) {  // proceedFront, both front Velodynes (and, in the built node, both rear ones: :378, :404)
  ProceedTable t;
  t.parts = {{p.vf_front_length, -p.roi_mid + p.vf_rear_length + p.vf_veh_length + p.vf_mid_length + p.vf_mid_length2, p.vf_z_max_ground_front},
             {p.vf_mid_length2, -p.roi_mid + p.vf_rear_length + p.vf_veh_length + p.vf_mid_length, p.vf_z_max_ground_mid2},
             {p.vf_mid_length, -p.roi_mid + p.vf_rear_length + p.vf_veh_length, p.vf_z_max_ground_mid},
             {p.vf_veh_length, -p.roi_mid + p.vf_rear_length, p.vf_z_max_ground_veh},
             {p.vf_rear_length, -p.roi_mid, p.vf_z_max_ground_rear}};
  return t;
}
inline ProceedTable rearTable(const Params& p) {  // proceedRear (:277-312; defined in the reference, never called)
  ProceedTable t;
  t.parts = {{p.vr_front_length, -p.roi_mid + p.vr_rear_length + p.vr_veh_length + p.vr_mid_length, p.vr_z_max_ground_front},
             {p.vr_mid_length, -p.roi_mid + p.vr_rear_length + p.vr_veh_length, p.vr_z_max_ground_mid},
             {p.vr_veh_length, -p.roi_mid + p.vr_rear_length, p.vr_z_max_ground_veh},
             {p.vr_rear_length, -p.roi_mid, p.vr_z_max_ground_rear}};
  return t;
}
inline ProceedTable topTable(const Params& p) {  // callbackTopMiddle (:428-446)
  ProceedTable t;
  t.parts = {{p.vt_front_length, p.vt_deviation_start_point, p.vt_z_max_ground_front}};
  t.plain = {{p.roi_mid + p.vt_deviation_start_point, -p.roi_mid, 0.0f}};
  return t;
}
inline ProceedTable livoxTable(const Params& p) {  // callbackFrontMiddle (:474-497)
  ProceedTable t;
  t.parts = {{p.l_front_length, p.l_deviation_mid_point + p.l_rear_length + p.l_mid_length + p.l_mid2_length, p.l_z_max_ground_front},
             {p.l_mid2_length, p.l_deviation_mid_point + p.l_rear_length + p.l_mid_length, p.l_z_max_ground_mid2},
             {p.l_mid_length, p.l_deviation_mid_point + p.l_rear_length, p.l_z_max_ground_mid},
             {p.l_rear_length, p.l_deviation_mid_point, p.l_z_max_ground_rear}};
  return t;
}
// void proceedFront(const Cloud::Ptr cloud_ptr, Cloud::Ptr no_ground_ptr, Cloud::Ptr ground_ptr) -- :228-269 -- and its
// siblings: getROI, then the table's zones, then the plain parts appended to the no-ground cloud.
inline void proceedTable(Context& ctx, const Cloud::Ptr& cloud_ptr, const ProceedTable& table, const Cloud::Ptr& no_ground_ptr,
                         const Cloud::Ptr& ground_ptr) {
  Cloud::Ptr cloud_ROI_ptr(new Cloud);
  getROI(ctx, cloud_ptr, cloud_ROI_ptr);
  proceedZones(ctx, cloud_ROI_ptr, table.parts, no_ground_ptr, ground_ptr, table.plain);
}
inline void proceedFront(Context& ctx, const Cloud::Ptr& c, const Cloud::Ptr& ng, const Cloud::Ptr& g) { proceedTable(ctx, c, frontTable(ctx.params()), ng, g); }
inline void proceedRear(Context& ctx, const Cloud::Ptr& c, const Cloud::Ptr& ng, const Cloud::Ptr& g) { proceedTable(ctx, c, rearTable(ctx.params()), ng, g); }
inline void proceedTop(Context& ctx, const Cloud::Ptr& c, const Cloud::Ptr& ng, const Cloud::Ptr& g) { proceedTable(ctx, c, topTable(ctx.params()), ng, g); }
inline void proceedLivox(Context& ctx, const Cloud::Ptr& c, const Cloud::Ptr& ng, const Cloud::Ptr& g) { proceedTable(ctx, c, livoxTable(ctx.params()), ng, g); }

// ---- my_cloud_fusion's variant of the same path (CloudFusionNode.h) -----------------------------------------------------------
// Its constants are double; every limit is narrowed to float where pcl::PassThrough::setFilterLimits(const float&, const
// float&) takes it, after the double arithmetic the reference writes (e.g. `mid_length/2 + front_length`).
inline cm_pass_t fpass(int axis, double lo, double hi) { return cm_pass_t{axis, static_cast<float>(lo), static_cast<float>(hi), 0}; }

// void filter_ROI_R(cloud, front, mid, rear, front_length, mid_length, rear_length) -- CloudFusionNode.h:145-190: z window,
// lane window in y, then three x ranges. The rear range is the reference's own [-(mid/2) - rear, rear] (its upper limit is
// `rear_length`, not `-mid_length/2`): reproduced as written.
inline void filter_ROI_R(Context& ctx, const FusionParams& fp, const Cloud::Ptr& cloud_ptr, const Cloud::Ptr& front_cloud_ptr,
                         const Cloud::Ptr& mid_cloud_ptr, const Cloud::Ptr& rear_cloud_ptr, const double front_length,
                         const double mid_length, const double rear_length) {
  const cm_pass_t z = fpass(2, fp.z_min, fp.z_max), y = fpass(1, -fp.lane_width / 2, fp.lane_width / 2);
  std::vector<cm_zone_t> zones(3);
  const cm_pass_t xr[3] = {fpass(0, mid_length / 2, (mid_length / 2) + front_length), fpass(0, -mid_length / 2, mid_length / 2),
                           fpass(0, -(mid_length / 2) - rear_length, rear_length)};
  for (int k = 0; k < 3; ++k) { zones[k].n_pass = 3; zones[k].pass[0] = z; zones[k].pass[1] = y; zones[k].pass[2] = xr[k]; }
  std::vector<Cloud> out;
  ctx.zone_split(*cloud_ptr, zones, out);
  *front_cloud_ptr = out[0]; *mid_cloud_ptr = out[1]; *rear_cloud_ptr = out[2];
}
// void filter_ROI_T(cloud, filtered) -- CloudFusionNode.h:87-143: the T shape = longitudinal bar += transverse bar
inline void filter_ROI_T(Context& ctx, const FusionParams& fp, const Cloud::Ptr& cloud_ptr, const Cloud::Ptr& filtered_cloud_ptr) {
  std::vector<cm_zone_t> zones(2);
  zones[0].n_pass = 3;
  zones[0].pass[0] = fpass(0, -fp.x_longitudinal / 2, fp.x_longitudinal / 2);
  zones[0].pass[1] = fpass(1, -fp.y_longitudinal / 2, fp.y_longitudinal / 2);
  zones[0].pass[2] = fpass(2, fp.z_min, fp.z_max);
  zones[1].n_pass = 3;
  zones[1].pass[0] = fpass(0, fp.x_longitudinal / 2, (fp.x_longitudinal / 2) + fp.x_transverse);
  zones[1].pass[1] = fpass(1, -fp.y_transverse / 2, fp.y_transverse / 2);
  zones[1].pass[2] = fpass(2, fp.z_min, fp.z_max);
  std::vector<Cloud> out;
  ctx.zone_split(*cloud_ptr, zones, out);
  Cloud first_part = out[0];
  first_part += out[1];
  *filtered_cloud_ptr = first_part;
}
// void remove_ground(cloud, no_ground, ground, z_min_ground, z_max_ground, max_angle) -- CloudFusionNode.h:192-216: in this
// package the RANSAC block is commented out (:219-271), so the function IS its two z windows.
inline void remove_ground(Context& ctx, const FusionParams& fp, const Cloud::Ptr& cloud_ptr, const Cloud::Ptr& no_ground_cloud_ptr,
                          const Cloud::Ptr& ground_cloud_ptr, const double z_min_ground, const double z_max_ground,
                          const double /*max_angle*/) {
  std::vector<cm_zone_t> zones(2);
  zones[0].n_pass = 1; zones[0].pass[0] = fpass(2, z_min_ground, z_max_ground);
  zones[1].n_pass = 1; zones[1].pass[0] = fpass(2, z_max_ground + 0.01, fp.z_max);
  std::vector<Cloud> out;
  ctx.zone_split(*cloud_ptr, zones, out);
  *ground_cloud_ptr = out[0];
  *no_ground_cloud_ptr = out[1];
}
// void remove_outliers(cloud) -- CloudFusionNode.h:74-85 (radius 0.1 m in this package)
inline void remove_outliers(Context& ctx, const FusionParams& fp, const Cloud::Ptr& cloud_ptr) {
  Cloud tmp;
  ctx.radius_outlier(*cloud_ptr, tmp, fp.radius, static_cast<int>(fp.min_neighbor));
  *cloud_ptr = tmp;
}
// proceed_pointcloud after the member-cloud copy (CloudFusionNode.h:327-493): filter_ROI_R, three remove_ground calls, the
// ground / no-ground parts appended front, mid, rear. `group`: 0 front Velodynes, 1 rear, 2 top, 3 Livox (index 0-1, 2-3, 4, 5).
// One zone-slicing pass: six chains of z, y, x-range, z-window.
inline void proceed_pointcloud(Context& ctx, const FusionParams& fp, const Cloud::Ptr& cloud_ptr, const Cloud::Ptr& no_ground_cloud_ptr,
                               const Cloud::Ptr& ground_cloud_ptr, int group) {
  const FusionParams::Group& g = fp.group[group];
  const cm_pass_t z = fpass(2, fp.z_min, fp.z_max), y = fpass(1, -fp.lane_width / 2, fp.lane_width / 2);
  const cm_pass_t xr[3] = {fpass(0, g.mid_length / 2, (g.mid_length / 2) + g.front_length), fpass(0, -g.mid_length / 2, g.mid_length / 2),
                           fpass(0, -(g.mid_length / 2) - g.rear_length, g.rear_length)};
  const double zlo[3] = {g.z_min_ground_front, g.z_min_ground_mid, g.z_min_ground_rear};
  const double zhi[3] = {g.z_max_ground_front, g.z_max_ground_mid, g.z_max_ground_rear};
  std::vector<cm_zone_t> zones(6);
  for (int k = 0; k < 3; ++k) {
    for (int w = 0; w < 2; ++w) {
      cm_zone_t& zn = zones[static_cast<size_t>(2 * k + w)];
      zn.n_pass = 4; zn.pass[0] = z; zn.pass[1] = y; zn.pass[2] = xr[k];
      zn.pass[3] = w == 0 ? fpass(2, zlo[k], zhi[k]) : fpass(2, zhi[k] + 0.01, fp.z_max);
    }
  }
  std::vector<Cloud> out;
  ctx.zone_split(*cloud_ptr, zones, out);
  Cloud ground1 = out[0], noground1 = out[1];
  ground1 += out[2]; ground1 += out[4];
  noground1 += out[3]; noground1 += out[5];
  *ground_cloud_ptr = ground1;
  *no_ground_cloud_ptr = noground1;
}

// void voxelgrid(const Cloud::Ptr cloud_ptr, Cloud::Ptr voxel_cloud_ptr) -- :168-177
inline void voxelgrid(Context& ctx, const Cloud::Ptr& cloud_ptr, const Cloud::Ptr& voxel_cloud_ptr) {
  Cloud tmp;
  ctx.voxelgrid(*cloud_ptr, tmp);
  *voxel_cloud_ptr = tmp;
}

// ---- the fused per-frame flow: callbacks submit, the main loop merges ------------------------------------------------------
// Replaces, together: callbackX (transform + ROI crop) -> member clouds / globals + flags -> concat -> voxelgrid, i.e. the
// merge of my_cloud_fusion's cloud_fusion() (CloudFusionNode.h:59-72, 506-534) with a crop, and the transform / getROI /
// fusePointclouds / voxelgrid skeleton of pcl_preprocessing (pc_preprocessing_main.cpp:318-337, :131-177, :574-578). It does
// NOT run the per-zone ground removal and outlier removal that pcl_preprocessing's callbacks do between getROI and the
// hand-off (proceedX): its voxel cloud is the VoxelGrid of the merged ROI cloud, not /points_voxel of that node. The whole
// main-loop iteration of pcl_preprocessing is PreprocessingFrame below.
// One GPU pass per frame instead of ~20 CPU passes.
class FusedFrame {
 public:
  FusedFrame(int n_sensors, int64_t max_points_per_sensor, uint64_t required_mask, int device = 0, Params p = Params(),
             bool first_cloud_wins = true)
      : params_(p), n_sensors_(n_sensors), required_(required_mask), cap_(max_points_per_sensor * n_sensors) {
    cm_config_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.device = device; cfg.max_sensors = n_sensors; cfg.max_points_per_sensor = max_points_per_sensor;
    cfg.max_point_step = 32; cfg.frames_in_flight = 2; cfg.max_batch_frames = 1; cfg.out_point_step = 32;
    if (cm_create(&cfg, &h_) != CM_OK) h_ = nullptr;
    if (h_) {
      const cm_pass_t passes[3] = {{2, p.roi_z_min, p.roi_z_max, 0}, {1, -p.roi_width / 2, p.roi_width / 2, 0},
                                   {0, -p.roi_mid, p.roi_length - p.roi_mid, 0}};
      cm_set_crop(h_, 3, passes);
      const float leaf[3] = {p.voxel_size, p.voxel_size, p.voxel_size};
      cm_set_voxel(h_, leaf, p.points_per_voxel, 1);
      cm_set_overflow_mode(h_, 1);  // behave like PCL when the leaf is too small
      // pcl_preprocessing keeps the FIRST cloud of a sensor after a fusion (`if (!flag_x)`, :330); my_cloud_fusion the newest
      cm_set_submit_policy(h_, first_cloud_wins ? CM_SUBMIT_FIRST_WINS : CM_SUBMIT_LATEST_WINS);
    }
  }
  ~FusedFrame() { if (h_) cm_destroy(h_); }
  FusedFrame(const FusedFrame&) = delete;
  FusedFrame& operator=(const FusedFrame&) = delete;
  bool ok() const { return h_ != nullptr; }
  cm_handle_t handle() const { return h_; }

  // once, after the TF lookup (pc_preprocessing_main.cpp:551-568)
  void setTransform(int sensor, const Transform& tf) { if (h_) cm_set_extrinsic_tf(h_, sensor, tf.q, tf.origin); }

  // body of callbackFrontRight ... callbackFrontMiddle: hands the raw cloud over. Safe to call from the six
  // ros::AsyncSpinner threads at once (pc_preprocessing_main.cpp:513) and concurrently with fuseAndVoxel: the hand-off
  // (submit + flag) and the main loop's (check + merge + flag reset) exclude each other -- the reference's own globals and
  // bool flags (pc_preprocessing_main.h:41-77) carry no such protection.
  void onCloud(int sensor, const Cloud& input) {
    const cm_layout_t l = pcl_layout(input.is_dense);
    onRecords(sensor, input.points.data(), static_cast<int64_t>(input.points.size()), l, stamp_of(input));
  }
  // the same for raw records in any PointCloud2 layout (msg.data as it arrived)
  void onRecords(int sensor, const void* data, int64_t n_points, const cm_layout_t& layout, uint64_t stamp) {
    if (!h_ || sensor < 0 || sensor >= n_sensors_) return;
    std::lock_guard<std::mutex> lk(gate_);
    if (cm_submit_cloud(h_, sensor, data, n_points, &layout, stamp) == CM_OK)
      seen_.fetch_or(1ull << sensor, std::memory_order_release);
  }
#ifdef CM_SHIM_HAVE_ROS_MSG
  // subscriber callback on the wire type: no pcl::PointCloud deserialisation, no by-value cloud copy
  bool onCloudMsg(int sensor, const sensor_msgs::PointCloud2& msg) {
    cm_layout_t l;
    if (layoutFromMsg(msg, &l) != CM_OK) return false;
    const uint64_t stamp = static_cast<uint64_t>(msg.header.stamp.sec) * 1000000ull + msg.header.stamp.nsec / 1000u;  // pcl_conversions::toPCL
    onRecords(sensor, msg.data.data(), static_cast<int64_t>(msg.width) * msg.height, l, stamp);
    return true;
  }
#endif
#ifdef CM_SHIM_HAVE_EIGEN
  void setTransform(int sensor, const Eigen::Matrix4f& m) { if (h_) setExtrinsic(h_, sensor, m); }
#endif
  // every required sensor has delivered since the last fusion (lock-free; the reference's `if (flag_a && flag_b ...)`, :134)
  bool ready() const { return (seen_.load(std::memory_order_acquire) & required_) == required_; }

  // fusePointclouds + voxelgrid. Returns false (like the reference's flag gate, :134) until every required sensor has
  // delivered; optional sensors are merged when present.
  bool fuseAndVoxel(Cloud& fused, Cloud& voxel) {
    if (!h_) return false;
    int64_t ticket = 0;
    {
      // check, enqueue and flag reset are one step with respect to the callbacks; the wait for the GPU happens outside
      std::lock_guard<std::mutex> lk(gate_);
      if (!ready()) return false;
      const int rc = cm_merge_frame_async(h_, ~0ull, &ticket);
      seen_.store(0, std::memory_order_release);  // every submission ends with the merge (consumed or discarded)
      if (rc != CM_OK) { fused.points.clear(); voxel.points.clear(); return false; }
    }
    fused.points.resize(static_cast<size_t>(cap_));
    voxel.points.resize(static_cast<size_t>(cap_));
    sx_.resize(static_cast<size_t>(cap_) * 4);
    cm_frame_out_t o;
    std::memset(&o, 0, sizeof(o));
    o.voxel_xyzi = voxel.points.data(); o.voxel_capacity = cap_;
    o.survivor_xyzi = sx_.data(); o.survivor_capacity = cap_;
    uint64_t used = 0, stamp = 0;
    const int rc = cm_wait_frame(h_, ticket, &o, &used, &stamp);
    if (rc != CM_OK) { fused.points.clear(); voxel.points.clear(); return false; }
    fused.points.resize(static_cast<size_t>(o.n_survivors));
    for (int64_t i = 0; i < o.n_survivors; ++i) {
      PointXYZI& p = fused.points[static_cast<size_t>(i)];
      p = PointXYZI();
      p.x = sx_[i * 4 + 0]; p.y = sx_[i * 4 + 1]; p.z = sx_[i * 4 + 2]; p.intensity = sx_[i * 4 + 3];
    }
    voxel.points.resize(static_cast<size_t>(o.n_voxels));
    for (Cloud* c : {&fused, &voxel}) {
      c->width = static_cast<uint32_t>(c->points.size()); c->height = 1; c->is_dense = true; set_stamp(*c, stamp);
    }
    return true;
  }

 private:
  Params params_;
  int n_sensors_;
  uint64_t required_;
  std::atomic<uint64_t> seen_{0};
  std::mutex gate_;
  int64_t cap_;
  cm_handle_t h_ = nullptr;
  std::vector<float> sx_;
};

// ---- one whole main-loop iteration of pcl_preprocessing, device-resident ----------------------------------------------------
// Replaces callbackX (transformPointCloud + proceedX: getROI, zones, removeGround per zone) -> globals + flags ->
// fusePointclouds -> voxelgrid -> the three published clouds (pc_preprocessing_main.cpp:318-508, :228-312, :131-177, :574-578).
// Each sensor has its own lane (handle + CUDA stream), so the six callbacks run concurrently like the reference's on
// ros::AsyncSpinner(6); a lane keeps the sensor's (no_ground, ground) clouds IN DEVICE MEMORY the way the reference keeps them
// in its globals: stored when the sensor's flag is clear (`if (!flag_x)`, :330), appended by every fusion -- also when stale or
// still empty, which is what happens to the optional top sensor there (:134-149) --, flags cleared by the fusion.
class PreprocessingFrame {
 public:
  // tables[s]: the zone table of sensor s (frontTable / rearTable / topTable / livoxTable)
  PreprocessingFrame(const std::vector<ProceedTable>& tables, int64_t max_points_per_sensor, uint64_t required_mask, int device = 0,
                     Params p = Params())
      : params_(p), required_(required_mask), cap_(max_points_per_sensor) {
    const int S = static_cast<int>(tables.size());
    lanes_.resize(static_cast<size_t>(S));
    ok_ = S > 0 && S <= 64;
    for (int s = 0; s < S && ok_; ++s) {
      Lane& l = *(lanes_[static_cast<size_t>(s)] = std::unique_ptr<Lane>(new Lane));
      cm_config_t cfg;
      std::memset(&cfg, 0, sizeof(cfg));
      cfg.device = device; cfg.max_sensors = 1; cfg.max_points_per_sensor = max_points_per_sensor; cfg.max_point_step = 32;
      cfg.max_batch_points = max_points_per_sensor; cfg.max_batch_frames = CM_MAX_PROCEED_PARTS; cfg.out_point_step = 32;
      ok_ = cm_create(&cfg, &l.h) == CM_OK;
      if (!ok_) { l.h = nullptr; break; }
      const cm_pass_t passes[3] = {{2, p.roi_z_min, p.roi_z_max, 0}, {1, -p.roi_width / 2, p.roi_width / 2, 0},
                                   {0, -p.roi_mid, p.roi_length - p.roi_mid, 0}};
      ok_ = cm_set_crop(l.h, 3, passes) == CM_OK && cm_stream_create(l.h, &l.stream) == CM_OK &&
            cm_dev_alloc(l.h, &l.raw, static_cast<size_t>(max_points_per_sensor) * 32 + 64) == CM_OK;
      l.cfg = proceedConfig(p, tables[static_cast<size_t>(s)].parts, tables[static_cast<size_t>(s)].plain);
    }
    if (ok_) {
      cm_config_t cfg;
      std::memset(&cfg, 0, sizeof(cfg));
      cfg.device = device; cfg.max_sensors = 1; cfg.max_points_per_sensor = 2 * max_points_per_sensor * S; cfg.max_point_step = 32;
      cfg.max_batch_points = 2 * max_points_per_sensor * S; cfg.max_batch_frames = 1; cfg.out_point_step = 32;
      ok_ = cm_create(&cfg, &voxel_) == CM_OK;
      if (!ok_) voxel_ = nullptr;
      const float leaf[3] = {p.voxel_size, p.voxel_size, p.voxel_size};
      const size_t bytes = static_cast<size_t>(2 * max_points_per_sensor * S) * 16 + 64;
      ok_ = ok_ && cm_set_voxel(voxel_, leaf, p.points_per_voxel, 1) == CM_OK && cm_dev_alloc(voxel_, &fused_ng_, bytes) == CM_OK &&
            cm_dev_alloc(voxel_, &fused_g_, bytes) == CM_OK;
    }
  }
  ~PreprocessingFrame() {
    for (auto& lp : lanes_) {
      if (!lp || !lp->h) continue;
      if (lp->stream) cm_stream_destroy(lp->h, lp->stream);
      if (lp->raw) cm_dev_free(lp->h, lp->raw);
      cm_destroy(lp->h);
    }
    if (voxel_) {
      if (fused_ng_) cm_dev_free(voxel_, fused_ng_);
      if (fused_g_) cm_dev_free(voxel_, fused_g_);
      cm_destroy(voxel_);
    }
  }
  PreprocessingFrame(const PreprocessingFrame&) = delete;
  PreprocessingFrame& operator=(const PreprocessingFrame&) = delete;
  bool ok() const { return ok_; }

  void setTransform(int sensor, const Transform& tf) {
    if (ok_ && sensor >= 0 && sensor < static_cast<int>(lanes_.size())) cm_set_extrinsic_tf(lanes_[static_cast<size_t>(sensor)]->h, 0, tf.q, tf.origin);
  }

  // body of callbackFrontRight ... callbackFrontMiddle: transform, proceedX, hand-off. One thread per sensor at a time.
  bool onCloud(int sensor, const Cloud& input) {
    if (!ok_ || sensor < 0 || sensor >= static_cast<int>(lanes_.size())) return false;
    Lane& l = *lanes_[static_cast<size_t>(sensor)];
    std::lock_guard<std::mutex> lk(l.mu);
    // `if (!flag_x) { store; flag_x = true; }`: the reference computes first and drops afterwards; skipping the work is the
    // same observable behaviour
    if (seen_.load(std::memory_order_acquire) & (1ull << sensor)) return true;
    const int64_t n = static_cast<int64_t>(input.points.size());
    if (n > cap_) return false;
    if (n && cm_memcpy_h2d(l.h, l.raw, input.points.data(), static_cast<size_t>(n) * 32, l.stream) != CM_OK) return false;
    cm_segment_t seg;
    seg.data = l.raw; seg.n_points = n; seg.layout = pcl_layout(input.is_dense); seg.sensor = 0; seg.frame = 0;
    cm_stats_t st;
    cm_device_out_t o;
    if (cm_dev_transform_crop(l.h, &seg, 1, l.stream) != CM_OK || cm_get_stats(l.h, &st) != CM_OK || cm_get_device_out(l.h, &o) != CM_OK)
      return false;
    cm_proceed_out_t po;
    if (cm_dev_proceed_zones(l.h, o.survivor_xyzi, st.survivors, &l.cfg, &po, l.stream) != CM_OK) return false;
    if (cm_stream_sync(l.h, l.stream) != CM_OK) return false;
    l.out = po;
    l.stamp = stamp_of(input);
    seen_.fetch_or(1ull << sensor, std::memory_order_release);
    return true;
  }

  bool ready() const { return (seen_.load(std::memory_order_acquire) & required_) == required_; }

  // fusePointclouds + voxelgrid + what publishPointcloud is handed: /points_no_ground, /points_ground, /points_voxel
  bool fuseAndVoxel(Cloud& no_ground, Cloud& ground, Cloud& voxel) {
    if (!ok_ || !ready()) return false;
    int64_t n_ng = 0, n_g = 0;
    uint64_t stamp = 0;
    for (auto& lp : lanes_) {  // sensor order; every lane's STORED clouds, fresh or not (the reference's globals)
      Lane& l = *lp;
      std::lock_guard<std::mutex> lk(l.mu);
      if (l.out.n_no_ground && cm_memcpy_d2d(voxel_, static_cast<char*>(fused_ng_) + n_ng * 16, l.out.no_ground_xyzi,
                                             static_cast<size_t>(l.out.n_no_ground) * 16, nullptr) != CM_OK) return false;
      if (l.out.n_ground && cm_memcpy_d2d(voxel_, static_cast<char*>(fused_g_) + n_g * 16, l.out.ground_xyzi,
                                          static_cast<size_t>(l.out.n_ground) * 16, nullptr) != CM_OK) return false;
      if (cm_stream_sync(voxel_, nullptr) != CM_OK) return false;  // the lane may be overwritten once its lock is released
      n_ng += l.out.n_no_ground; n_g += l.out.n_ground;
      if (l.stamp > stamp) stamp = l.stamp;
    }
    seen_.store(0, std::memory_order_release);
    cm_stats_t st;
    cm_device_out_t o;
    if (cm_dev_voxelgrid(voxel_, static_cast<const float*>(fused_ng_), n_ng, 1, nullptr) != CM_OK || cm_get_stats(voxel_, &st) != CM_OK ||
        cm_get_device_out(voxel_, &o) != CM_OK)
      return false;
    auto fetch = [&](Cloud& c, const void* dev, int64_t n) {
      buf_.resize(static_cast<size_t>(n) * 4 + 4);
      if (n && cm_memcpy_d2h(voxel_, buf_.data(), dev, static_cast<size_t>(n) * 16, nullptr) != CM_OK) return false;
      c.points.resize(static_cast<size_t>(n));
      for (int64_t i = 0; i < n; ++i) {
        PointXYZI& p = c.points[static_cast<size_t>(i)];
        p = PointXYZI();
        p.x = buf_[i * 4 + 0]; p.y = buf_[i * 4 + 1]; p.z = buf_[i * 4 + 2]; p.intensity = buf_[i * 4 + 3];
      }
      return true;
    };
    if (!fetch(no_ground, fused_ng_, n_ng) || !fetch(ground, fused_g_, n_g)) return false;
    if (st.pcl_overflow) {
      voxel = no_ground;  // PCL 1.8.1: leaf too small -> output = input
    } else {
      voxel.points.resize(static_cast<size_t>(st.voxels_out));
      if (st.voxels_out && cm_memcpy_d2h(voxel_, voxel.points.data(), o.voxel_xyzi, static_cast<size_t>(st.voxels_out) * 32, nullptr) != CM_OK)
        return false;
    }
    for (Cloud* c : {&no_ground, &ground, &voxel}) {
      c->width = static_cast<uint32_t>(c->points.size()); c->height = 1; c->is_dense = true; set_stamp(*c, stamp);
    }
    return true;
  }

 private:
  struct Lane {
    cm_handle_t h = nullptr;
    void* stream = nullptr;
    void* raw = nullptr;
    cm_proceed_cfg_t cfg;
    cm_proceed_out_t out;
    uint64_t stamp = 0;
    std::mutex mu;
    Lane() { std::memset(&cfg, 0, sizeof(cfg)); std::memset(&out, 0, sizeof(out)); }
  };
  Params params_;
  uint64_t required_;
  std::atomic<uint64_t> seen_{0};
  int64_t cap_;
  bool ok_ = false;
  std::vector<std::unique_ptr<Lane>> lanes_;
  cm_handle_t voxel_ = nullptr;
  void *fused_ng_ = nullptr, *fused_g_ = nullptr;
  std::vector<float> buf_;
};

}  // namespace cloud_merger

#endif  // CLOUD_MERGER_SHIM_HPP_
