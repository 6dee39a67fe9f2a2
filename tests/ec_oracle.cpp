/*
 * ec_oracle.cpp -- CPU oracle of pcl::EuclideanClusterExtraction (TEST INFRASTRUCTURE ONLY): PCL 1.8.1's loop
 * (segmentation/impl/extract_clusters.hpp, extractEuclideanClusters with a KdTreeFLANN) stated literally, built by
 * tests/ec_oracle.py with the flags of oracle/Makefile (-O2 -ffp-contract=off, no -march, no -ffast-math): every float
 * multiply and add rounds on its own.
 *
 * PCL 1.8.1, in substance:
 *   extract():  extractEuclideanClusters(*input_, *indices_, tree_, static_cast<float>(cluster_tolerance_), clusters,
 *                                        min_pts_per_cluster_, max_pts_per_cluster_);
 *   radiusSearch(i, radius, ...) with that float widened to double: FLANN gets static_cast<float>(radius * radius) and
 *   returns every point whose L2_Simple float distance (dx*dx + dy*dy) + dz*dz is strictly below it, sorted by
 *   (distance, index);
 *   for (i = 0; i < n; ++i) {
 *     if (processed[i]) continue;
 *     seed_queue = {i}; processed[i] = true;
 *     for (sq_idx = 0; sq_idx < seed_queue.size(); ++sq_idx) {
 *       if (!tree->radiusSearch(seed_queue[sq_idx], tolerance, nn_indices, nn_distances)) continue;
 *       for (j = 1; j < nn_indices.size(); ++j)           // nn_start_idx = 1
 *         if (!processed[nn_indices[j]]) { seed_queue.push_back(nn_indices[j]); processed[nn_indices[j]] = true; }
 *     }
 *     if (min_pts <= seed_queue.size() <= max_pts) { r.indices = seed_queue; std::sort(r.indices); clusters.push_back(r); }
 *   }
 *   std::sort(clusters.rbegin(), clusters.rend(), comparePointClusters);   // a.indices.size() < b.indices.size()
 * The neighbour lists are those of an exhaustive search; a grid of cells twice the tolerance wide, indexed in double,
 * only narrows the candidates (a neighbour is at most one such cell away on every axis). Non-finite points are skipped
 * (PCL would search from them; the library's documented deviation).
 */
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <unordered_map>
#include <utility>
#include <vector>

namespace {

struct CellHash {
  size_t operator()(const std::pair<int64_t, int64_t>& k) const {
    return std::hash<int64_t>()(k.first * 1000003 + k.second);
  }
};

struct Cluster {
  std::vector<int64_t> indices;
};
bool comparePointClusters(const Cluster& a, const Cluster& b) { return a.indices.size() < b.indices.size(); }

}  // namespace

extern "C" {

/* xyzi: n points of 4 floats. idx_out[n], begin_out[n + 1]: the clusters in PCL's order; *n_clusters. */
int cmo_euclidean_clusters(const float* xyzi, int64_t n, double tolerance, int32_t min_size, int32_t max_size,
                           int64_t* idx_out, int64_t* begin_out, int64_t* n_clusters) {
  if (n < 0) return 1;
  const float tf = static_cast<float>(tolerance);
  const double radius = tf;
  const float r2 = static_cast<float>(radius * radius);
  const double cell = 2.0 * radius;
  auto fin = [&](int64_t i) {
    const float* p = xyzi + 4 * i;
    return std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]);
  };
  auto cix = [&](float v) { return (int64_t)std::floor((double)v / cell); };
  // cells keyed by (x, y) index pair and z index: (x * 2^21 + y, z)
  std::unordered_map<std::pair<int64_t, int64_t>, std::vector<int64_t>, CellHash> grid;
  auto key_of = [&](int64_t cx, int64_t cy, int64_t cz) { return std::make_pair(cx * 2097152 + cy, cz); };
  for (int64_t i = 0; i < n; ++i)
    if (fin(i)) grid[key_of(cix(xyzi[4 * i]), cix(xyzi[4 * i + 1]), cix(xyzi[4 * i + 2]))].push_back(i);
  std::vector<std::pair<float, int64_t>> nn;
  auto radius_search = [&](int64_t q) {
    nn.clear();
    const float* a = xyzi + 4 * q;
    const int64_t cx = cix(a[0]), cy = cix(a[1]), cz = cix(a[2]);
    for (int64_t dx = -1; dx <= 1; ++dx)
      for (int64_t dy = -1; dy <= 1; ++dy)
        for (int64_t dz = -1; dz <= 1; ++dz) {
          auto it = grid.find(key_of(cx + dx, cy + dy, cz + dz));
          if (it == grid.end()) continue;
          for (int64_t j : it->second) {
            const float* b = xyzi + 4 * j;
            const float ex = a[0] - b[0], ey = a[1] - b[1], ez = a[2] - b[2];
            const float xx = ex * ex, yy = ey * ey, zz = ez * ez;
            const float s = xx + yy;
            const float d = s + zz;
            if (d < r2) nn.push_back(std::make_pair(d, j));
          }
        }
    std::sort(nn.begin(), nn.end());
  };
  std::vector<bool> processed((size_t)n, false);
  std::vector<Cluster> clusters;
  for (int64_t i = 0; i < n; ++i) {
    if (processed[i] || !fin(i)) continue;
    std::vector<int64_t> seed_queue;
    size_t sq_idx = 0;
    seed_queue.push_back(i);
    processed[i] = true;
    while (sq_idx < seed_queue.size()) {
      radius_search(seed_queue[sq_idx]);
      if (nn.empty()) { sq_idx++; continue; }
      for (size_t j = 1; j < nn.size(); ++j) {
        if (processed[nn[j].second]) continue;
        seed_queue.push_back(nn[j].second);
        processed[nn[j].second] = true;
      }
      sq_idx++;
    }
    if (seed_queue.size() >= (size_t)min_size && seed_queue.size() <= (size_t)max_size) {
      Cluster r;
      r.indices = seed_queue;
      std::sort(r.indices.begin(), r.indices.end());
      clusters.push_back(r);
    }
  }
  std::sort(clusters.rbegin(), clusters.rend(), comparePointClusters);
  int64_t at = 0;
  begin_out[0] = 0;
  for (size_t c = 0; c < clusters.size(); ++c) {
    for (int64_t v : clusters[c].indices) idx_out[at++] = v;
    begin_out[c + 1] = at;
  }
  *n_clusters = (int64_t)clusters.size();
  return 0;
}

/* The order std::sort(v.rbegin(), v.rend(), size <) leaves k clusters of the given sizes in: order_out[r] = the input
 * position of the cluster at rank r. */
int cmo_pcl_cluster_order(const int64_t* sizes, int64_t k, int64_t* order_out) {
  std::vector<std::pair<int64_t, int64_t>> v((size_t)k);
  for (int64_t i = 0; i < k; ++i) v[i] = std::make_pair(sizes[i], i);
  std::sort(v.rbegin(), v.rend(), [](const std::pair<int64_t, int64_t>& a, const std::pair<int64_t, int64_t>& b) {
    return a.first < b.first;
  });
  for (int64_t i = 0; i < k; ++i) order_out[i] = v[i].second;
  return 0;
}

}  // extern "C"
