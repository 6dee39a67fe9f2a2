// plane_axis_pcl_ref.cpp -- the REAL pcl::SACSegmentation<PointXYZI> (SAC_RANSAC, any of SACMODEL_PLANE,
// SACMODEL_PERPENDICULAR_PLANE, SACMODEL_PARALLEL_PLANE) behind a C signature (TEST INFRASTRUCTURE ONLY), so that a machine
// with PCL (1.8.x, the ROS Melodic pin) can pin tests/plane_axis_oracle.cpp against the library itself.
// tests/plane_axis_oracle.py builds it with g++ and pkg-config where PCL is installed; tests/test_plane_axis_vs_pcl.py skips
// (and says why) where it is not.
#include <pcl/ModelCoefficients.h>
#include <pcl/PointIndices.h>
#include <pcl/point_cloud.h>
#include <pcl/point_types.h>
#include <pcl/sample_consensus/method_types.h>
#include <pcl/sample_consensus/model_types.h>
#include <pcl/segmentation/sac_segmentation.h>

#include <cstdint>

extern "C" {

// coeff_out[4]; out_inliers ascending; returns the number of inliers (0: segment() failed or kept none)
int64_t cmp_plane_ransac_model(const float* xyzi, int64_t n, double threshold, double probability, int32_t max_iterations,
                               int32_t optimize, int32_t model, const float* axis, double eps_angle, float* coeff_out,
                               int32_t* out_inliers) {
  pcl::PointCloud<pcl::PointXYZI>::Ptr in(new pcl::PointCloud<pcl::PointXYZI>);
  in->points.resize(static_cast<size_t>(n));
  for (int64_t i = 0; i < n; ++i) {
    pcl::PointXYZI& p = in->points[static_cast<size_t>(i)];
    p.x = xyzi[4 * i]; p.y = xyzi[4 * i + 1]; p.z = xyzi[4 * i + 2]; p.intensity = xyzi[4 * i + 3];
  }
  in->width = static_cast<uint32_t>(n);
  in->height = 1;
  in->is_dense = true;
  pcl::SACSegmentation<pcl::PointXYZI> seg;
  pcl::PointIndices::Ptr inliers(new pcl::PointIndices);
  pcl::ModelCoefficients::Ptr coefficients(new pcl::ModelCoefficients);
  seg.setModelType(model == 1 ? pcl::SACMODEL_PERPENDICULAR_PLANE : model == 2 ? pcl::SACMODEL_PARALLEL_PLANE : pcl::SACMODEL_PLANE);
  seg.setMethodType(pcl::SAC_RANSAC);
  seg.setMaxIterations(max_iterations);
  seg.setAxis(Eigen::Vector3f(axis[0], axis[1], axis[2]));
  seg.setEpsAngle(eps_angle);
  seg.setDistanceThreshold(threshold);
  seg.setOptimizeCoefficients(optimize != 0);
  seg.setProbability(probability);
  seg.setInputCloud(in);
  seg.segment(*inliers, *coefficients);
  for (size_t i = 0; i < inliers->indices.size(); ++i) out_inliers[i] = inliers->indices[i];
  if (coeff_out)
    for (size_t k = 0; k < 4; ++k) coeff_out[k] = k < coefficients->values.size() ? coefficients->values[k] : 0.0f;
  return static_cast<int64_t>(inliers->indices.size());
}

}  // extern "C"
