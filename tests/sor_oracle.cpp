/*
 * sor_oracle.cpp -- CPU oracle of pcl::StatisticalOutlierRemoval (TEST INFRASTRUCTURE ONLY): a restatement of PCL 1.8.1
 * StatisticalOutlierRemoval<PointXYZI>::applyFilterIndices (filters/impl/statistical_outlier_removal.hpp) with an
 * exhaustive neighbour search in place of FLANN's exact KDTreeSingleIndex, built by tests/sor_oracle.py with the flags of
 * oracle/Makefile (-O2 -ffp-contract=off, no -march, no -ffast-math): every float multiply and add rounds on its own.
 *
 * PCL 1.8.1, in substance (keep_organized false, indices_ = every point, searcher_ = KdTree<PointT>(false)):
 *   for iii: if (!isfinite(x) || !isfinite(y) || !isfinite(z)) { distances[iii] = 0; continue; }
 *            searcher_->nearestKSearch(iii, mean_k_ + 1, nn_indices, nn_dists);      // ascending; [0] = the point
 *            double dist_sum = 0; for (k = 1; k < mean_k_ + 1; ++k) dist_sum += sqrt(nn_dists[k]);
 *            distances[iii] = static_cast<float>(dist_sum / mean_k_); valid_distances++;
 *   double sum = 0, sq_sum = 0;
 *   for i: { sum += distances[i]; sq_sum += distances[i] * distances[i]; }           // float product
 *   mean = sum / valid; variance = (sq_sum - sum * sum / valid) / (valid - 1); stddev = sqrt(variance);
 *   distance_threshold = mean + std_mul_ * stddev;
 *   for iii: removed iff (!negative_ && distances[iii] > threshold) || (negative_ && distances[iii] <= threshold)
 * nn_dists are FLANN L2_Simple float distances, (dx*dx + dy*dy) + dz*dz. The unqualified sqrt is std::sqrt(float) or
 * ::sqrt(double) depending on the build: sqrt_mode 0 / 1. A cloud with 0 < valid <= mean_k makes PCL read past its
 * neighbour vectors (undefined); here every point of such a cloud is kept and its distances stay 0.
 */
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <vector>

extern "C" {

typedef struct {
  double mean, stddev, threshold, sum, sq_sum;
  int64_t n_valid;
  int32_t too_few;
  int32_t n_kept;
} cmo_sor_stats_t;

/* xyzi: n points of 4 floats. dist[n] out: PCL's distances[]; keep[n] out: 1 = kept. */
int cmo_statistical_outlier(const float* xyzi, int64_t n, int mean_k, double std_mul, int negative, int sqrt_mode,
                            float* dist, uint8_t* keep, cmo_sor_stats_t* st) {
  if (mean_k < 1 || n < 0) return 1;
  std::vector<int64_t> fin;
  for (int64_t i = 0; i < n; ++i) {
    const float* p = xyzi + 4 * i;
    if (std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2])) fin.push_back(i);
  }
  const int64_t valid = (int64_t)fin.size();
  const bool too_few = valid > 0 && valid <= mean_k;
  std::vector<float> d2((size_t)valid);
  for (int64_t i = 0; i < n; ++i) dist[i] = 0.0f;
  if (valid > 0 && !too_few) {
    for (int64_t a = 0; a < valid; ++a) {
      const float* q = xyzi + 4 * fin[a];
      for (int64_t b = 0; b < valid; ++b) {
        const float* p = xyzi + 4 * fin[b];
        const float dx = q[0] - p[0], dy = q[1] - p[1], dz = q[2] - p[2];
        const float xx = dx * dx, yy = dy * dy, zz = dz * dz;
        const float s = xx + yy;
        d2[b] = s + zz;
      }
      std::partial_sort(d2.begin(), d2.begin() + (mean_k + 1), d2.end());
      double dist_sum = 0.0;
      for (int k = 1; k < mean_k + 1; ++k) {
        if (sqrt_mode == 0) dist_sum += std::sqrt(d2[k]);              // std::sqrt(float), promoted
        else dist_sum += ::sqrt(static_cast<double>(d2[k]));          // ::sqrt(double)
      }
      dist[fin[a]] = static_cast<float>(dist_sum / mean_k);
    }
  }
  double sum = 0.0, sq_sum = 0.0;
  for (int64_t i = 0; i < n; ++i) {
    sum += dist[i];
    const float sq = dist[i] * dist[i];
    sq_sum += sq;
  }
  const double vd = static_cast<double>(valid);
  const double mean = sum / vd;
  const double p = sum * sum;
  const double q = p / vd;
  const double variance = (sq_sum - q) / (vd - 1.0);
  const double stddev = std::sqrt(variance);
  const double m = std_mul * stddev;
  const double threshold = mean + m;
  int32_t kept = 0;
  for (int64_t i = 0; i < n; ++i) {
    const bool removed = !too_few && ((!negative && dist[i] > threshold) || (negative && dist[i] <= threshold));
    keep[i] = removed ? 0 : 1;
    kept += removed ? 0 : 1;
  }
  st->mean = mean; st->stddev = stddev; st->threshold = threshold; st->sum = sum; st->sq_sum = sq_sum;
  st->n_valid = valid; st->too_few = too_few ? 1 : 0; st->n_kept = kept;
  return 0;
}

}  // extern "C"
