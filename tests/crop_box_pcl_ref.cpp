// crop_box_pcl_ref.cpp -- the REAL pcl::CropBox<PointXYZI> behind the C signature of cmo_crop_box (TEST INFRASTRUCTURE ONLY),
// so that a machine with PCL (1.8.x, the ROS Melodic pin) can pin tests/crop_box_oracle.cpp against the library itself.
// tests/crop_box_oracle.py builds it with g++ and pkg-config where PCL is installed; tests/test_crop_box_vs_pcl.py skips
// (and says why) where it is not.
#include <pcl/filters/crop_box.h>
#include <pcl/point_cloud.h>
#include <pcl/point_types.h>

#include <Eigen/Geometry>
#include <cstdint>
#include <vector>

extern "C" {

// box: the layout of cm_crop_box_t / cmo_crop_box_t (min[3], max[3], translation[3], rotation[3], transform[12]); the
// cloud's is_dense flag as given
int64_t cmp_crop_box(const float* xyzi, int64_t n, int32_t is_dense, const float* box24, int32_t negative, int32_t* out_idx) {
  pcl::PointCloud<pcl::PointXYZI>::Ptr in(new pcl::PointCloud<pcl::PointXYZI>);
  in->points.resize(static_cast<size_t>(n));
  for (int64_t i = 0; i < n; ++i) {
    pcl::PointXYZI& p = in->points[static_cast<size_t>(i)];
    p.x = xyzi[i * 4 + 0]; p.y = xyzi[i * 4 + 1]; p.z = xyzi[i * 4 + 2]; p.intensity = xyzi[i * 4 + 3];
  }
  in->width = static_cast<uint32_t>(n); in->height = 1; in->is_dense = is_dense != 0;
  pcl::CropBox<pcl::PointXYZI> cb;
  cb.setInputCloud(in);
  cb.setMin(Eigen::Vector4f(box24[0], box24[1], box24[2], 1.0f));
  cb.setMax(Eigen::Vector4f(box24[3], box24[4], box24[5], 1.0f));
  cb.setTranslation(Eigen::Vector3f(box24[6], box24[7], box24[8]));
  cb.setRotation(Eigen::Vector3f(box24[9], box24[10], box24[11]));
  Eigen::Affine3f t = Eigen::Affine3f::Identity();
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 4; ++c) t.matrix()(r, c) = box24[12 + r * 4 + c];
  cb.setTransform(t);
  cb.setNegative(negative != 0);
  std::vector<int> idx;
  cb.filter(idx);
  for (size_t i = 0; i < idx.size(); ++i) out_idx[i] = idx[i];
  return static_cast<int64_t>(idx.size());
}

}  // extern "C"
