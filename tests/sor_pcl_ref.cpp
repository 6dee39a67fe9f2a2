// sor_pcl_ref.cpp -- the REAL pcl::StatisticalOutlierRemoval<PointXYZI> behind a C signature (TEST INFRASTRUCTURE ONLY), so
// that a machine with PCL (1.8.x, the ROS Melodic pin) can pin tests/sor_oracle.cpp against the library itself.
// tests/sor_oracle.py builds it with g++ and pkg-config where PCL is installed; tests/test_sor_vs_pcl.py skips (and says
// why) where it is not. The cloud is passed as non-dense, as the GPU path treats every input.
#include <pcl/filters/statistical_outlier_removal.h>
#include <pcl/point_cloud.h>
#include <pcl/point_types.h>

#include <cstdint>
#include <vector>

extern "C" {

// indices of the kept points, in input order, into out_idx[n]; returns their number
int64_t cmp_statistical_outlier(const float* xyzi, int64_t n, int32_t mean_k, double std_mul, int32_t negative,
                                int32_t* out_idx) {
  pcl::PointCloud<pcl::PointXYZI>::Ptr in(new pcl::PointCloud<pcl::PointXYZI>);
  in->points.resize(static_cast<size_t>(n));
  for (int64_t i = 0; i < n; ++i) {
    pcl::PointXYZI& p = in->points[static_cast<size_t>(i)];
    p.x = xyzi[4 * i]; p.y = xyzi[4 * i + 1]; p.z = xyzi[4 * i + 2]; p.intensity = xyzi[4 * i + 3];
  }
  in->width = static_cast<uint32_t>(n);
  in->height = 1;
  in->is_dense = false;
  pcl::StatisticalOutlierRemoval<pcl::PointXYZI> sor;
  sor.setInputCloud(in);
  sor.setMeanK(mean_k);
  sor.setStddevMulThresh(std_mul);
  sor.setNegative(negative != 0);
  std::vector<int> kept;
  sor.filter(kept);
  for (size_t i = 0; i < kept.size(); ++i) out_idx[i] = kept[i];
  return static_cast<int64_t>(kept.size());
}

}  // extern "C"
