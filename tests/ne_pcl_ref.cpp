// ne_pcl_ref.cpp -- the REAL pcl::NormalEstimation<PointXYZI, Normal> with a KdTree and a radius search behind a C
// signature (TEST INFRASTRUCTURE ONLY), so that a machine with PCL (1.8.x, the ROS Melodic pin) can compare
// tests/ne_oracle.cpp with the library itself. tests/test_ne_vs_pcl.py builds it with g++ and pkg-config where PCL is
// installed and skips (and says why) where it is not.
#include <pcl/features/normal_3d.h>
#include <pcl/point_cloud.h>
#include <pcl/point_types.h>
#include <pcl/search/kdtree.h>

#include <cstdint>

extern "C" {

// out[n][4] = normal_x normal_y normal_z curvature of every input point
int cmp_normals(const float* xyzi, int64_t n, double radius, const float* vp, float* out) {
  pcl::PointCloud<pcl::PointXYZI>::Ptr in(new pcl::PointCloud<pcl::PointXYZI>);
  in->points.resize(static_cast<size_t>(n));
  for (int64_t i = 0; i < n; ++i) {
    pcl::PointXYZI& p = in->points[static_cast<size_t>(i)];
    p.x = xyzi[4 * i]; p.y = xyzi[4 * i + 1]; p.z = xyzi[4 * i + 2]; p.intensity = xyzi[4 * i + 3];
  }
  in->width = static_cast<uint32_t>(n);
  in->height = 1;
  in->is_dense = false;
  pcl::search::KdTree<pcl::PointXYZI>::Ptr tree(new pcl::search::KdTree<pcl::PointXYZI>);
  pcl::NormalEstimation<pcl::PointXYZI, pcl::Normal> ne;
  ne.setInputCloud(in);
  ne.setSearchMethod(tree);
  ne.setRadiusSearch(radius);
  ne.setViewPoint(vp[0], vp[1], vp[2]);
  pcl::PointCloud<pcl::Normal> normals;
  ne.compute(normals);
  for (int64_t i = 0; i < n; ++i) {
    const pcl::Normal& q = normals.points[static_cast<size_t>(i)];
    out[4 * i] = q.normal_x; out[4 * i + 1] = q.normal_y; out[4 * i + 2] = q.normal_z; out[4 * i + 3] = q.curvature;
  }
  return 0;
}

}  // extern "C"
