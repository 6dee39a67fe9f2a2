// test_shim_ec.cpp -- the Euclidean cluster extraction of the reference-facing shim (include/cloud_merger_shim.hpp):
// extractEuclideanClusters() and Context::euclidean_clusters[_multi] against the C++ statement of
// pcl::EuclideanClusterExtraction (tests/ec_oracle.cpp): the same clusters in the same order. Without a CUDA device it must
// refuse (exit 77).
#include <cmath>
#include <cstdio>
#include <limits>
#include <vector>

#include "cloud_merger_shim.hpp"

using namespace cloud_merger;

extern "C" int cmo_euclidean_clusters(const float* xyzi, int64_t n, double tolerance, int32_t min_size, int32_t max_size,
                                      int64_t* idx_out, int64_t* begin_out, int64_t* n_clusters);

static int g_fail = 0;
#define CHECK(cond, ...)                                   \
  do {                                                     \
    if (!(cond)) {                                         \
      std::printf("FAIL %s:%d: ", __FILE__, __LINE__);     \
      std::printf(__VA_ARGS__);                            \
      std::printf("\n");                                   \
      ++g_fail;                                            \
    }                                                      \
  } while (0)

static uint64_t g_rng = 0x2545F4914F6CDD1Dull;
static double urand() {  // splitmix64
  uint64_t z = (g_rng += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (z >> 11) * (1.0 / 9007199254740992.0);
}

static Cloud make_cloud(size_t n) {  // blobs of returns, a few strays, exact duplicates and NaN rows
  Cloud c;
  c.points.resize(n);
  for (size_t i = 0; i < n; ++i) {
    PointXYZI& p = c.points[i];
    const double cx = 3.0 * std::floor(8.0 * urand()), cy = 3.0 * std::floor(8.0 * urand());
    p.x = static_cast<float>(cx + 0.6 * urand());
    p.y = static_cast<float>(cy + 0.6 * urand());
    p.z = static_cast<float>(0.3 * urand());
    p.intensity = static_cast<float>(255.0 * urand());
    if (i > 0 && urand() < 0.05) p = c.points[i - 1];
    if (urand() < 0.01) p.y = std::numeric_limits<float>::quiet_NaN();
  }
  c.width = static_cast<uint32_t>(n); c.height = 1; c.is_dense = false;
  return c;
}

static void compare(const Cloud& in, const std::vector<std::vector<int>>& got, double tol, int mn, int mx, const char* what) {
  const size_t n = in.points.size();
  std::vector<float> xyzi(4 * n + 4);
  for (size_t i = 0; i < n; ++i) {
    xyzi[4 * i] = in.points[i].x; xyzi[4 * i + 1] = in.points[i].y;
    xyzi[4 * i + 2] = in.points[i].z; xyzi[4 * i + 3] = in.points[i].intensity;
  }
  std::vector<int64_t> idx(n + 1), begin(n + 1);
  int64_t k = 0;
  CHECK(cmo_euclidean_clusters(xyzi.data(), static_cast<int64_t>(n), tol, mn, mx, idx.data(), begin.data(), &k) == 0,
        "%s: oracle", what);
  bool same = static_cast<int64_t>(got.size()) == k;
  for (int64_t j = 0; same && j < k; ++j) {
    same = static_cast<int64_t>(got[j].size()) == begin[j + 1] - begin[j];
    for (int64_t t = begin[j]; same && t < begin[j + 1]; ++t) same = got[j][t - begin[j]] == idx[t];
  }
  CHECK(same, "%s: %zu clusters, oracle %lld", what, got.size(), static_cast<long long>(k));
  CHECK(k > 1, "%s: the case has several clusters", what);
}

int main() {
  if (cm_device_count() == 0) {
    std::printf("no CUDA device: the shim has no CPU path (expected on the build box)\n");
    Context ctx(1024);
    CHECK(!ctx.ok(), "Context must fail without a GPU");
    return g_fail ? 1 : 77;  // 77 = skipped
  }
  Context ctx(1 << 15, 2);
  CHECK(ctx.ok(), "Context: %s", ctx.last_error().c_str());
  const Cloud a = make_cloud(6000), b = make_cloud(3000);
  {  // the drop-in function
    Cloud::Ptr p(new Cloud(a));
    std::vector<std::vector<int>> clusters;
    extractEuclideanClusters(ctx, p, 0.5, 10, 25000, clusters);
    CHECK(ctx.ok(), "extractEuclideanClusters: %s", ctx.last_error().c_str());
    compare(a, clusters, 0.5, 10, 25000, "extractEuclideanClusters");
  }
  {  // two clouds in one call, a tolerance that is not a float
    std::vector<std::vector<std::vector<int>>> out;
    CHECK(ctx.euclidean_clusters_multi({&a, &b}, out, 0.1, 1, 2147483647), "multi: %s", ctx.last_error().c_str());
    CHECK(out.size() == 2, "multi: two results");
    if (out.size() == 2) {
      compare(a, out[0], 0.1, 1, 2147483647, "multi cloud 0");
      compare(b, out[1], 0.1, 1, 2147483647, "multi cloud 1");
    }
  }
  {  // the radius filter still runs on the same context afterwards
    Cloud out;
    CHECK(ctx.radius_outlier(a, out, 0.15, 1) && !out.points.empty(), "radius_outlier after: %s", ctx.last_error().c_str());
  }
  if (!g_fail) std::printf("shim ec ok\n");
  return g_fail ? 1 : 0;
}
