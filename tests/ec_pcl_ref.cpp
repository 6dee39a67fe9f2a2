// ec_pcl_ref.cpp -- the REAL pcl::EuclideanClusterExtraction<PointXYZI> with a KdTree behind a C signature (TEST
// INFRASTRUCTURE ONLY), so that a machine with PCL (1.8.x, the ROS Melodic pin) can pin tests/ec_oracle.cpp against the
// library itself. tests/ec_oracle.py builds it with g++ and pkg-config where PCL is installed; tests/test_ec_vs_pcl.py
// skips (and says why) where it is not. Only finite clouds are passed: PCL searches from non-finite points, which the
// library documents as a deviation.
#include <pcl/point_cloud.h>
#include <pcl/point_types.h>
#include <pcl/search/kdtree.h>
#include <pcl/segmentation/extract_clusters.h>

#include <cstdint>
#include <vector>

extern "C" {

// the clusters in PCL's order: their indices into idx_out[n], cluster j = [begin_out[j], begin_out[j+1]); returns their number
int64_t cmp_euclidean_clusters(const float* xyzi, int64_t n, double tolerance, int32_t min_size, int32_t max_size,
                               int64_t* idx_out, int64_t* begin_out) {
  pcl::PointCloud<pcl::PointXYZI>::Ptr in(new pcl::PointCloud<pcl::PointXYZI>);
  in->points.resize(static_cast<size_t>(n));
  for (int64_t i = 0; i < n; ++i) {
    pcl::PointXYZI& p = in->points[static_cast<size_t>(i)];
    p.x = xyzi[4 * i]; p.y = xyzi[4 * i + 1]; p.z = xyzi[4 * i + 2]; p.intensity = xyzi[4 * i + 3];
  }
  in->width = static_cast<uint32_t>(n);
  in->height = 1;
  pcl::search::KdTree<pcl::PointXYZI>::Ptr tree(new pcl::search::KdTree<pcl::PointXYZI>);
  tree->setInputCloud(in);
  std::vector<pcl::PointIndices> clusters;
  pcl::EuclideanClusterExtraction<pcl::PointXYZI> ec;
  ec.setClusterTolerance(tolerance);
  ec.setMinClusterSize(min_size);
  ec.setMaxClusterSize(max_size);
  ec.setSearchMethod(tree);
  ec.setInputCloud(in);
  ec.extract(clusters);
  int64_t at = 0;
  begin_out[0] = 0;
  for (size_t c = 0; c < clusters.size(); ++c) {
    for (int v : clusters[c].indices) idx_out[at++] = v;
    begin_out[c + 1] = at;
  }
  return static_cast<int64_t>(clusters.size());
}

}  // extern "C"
