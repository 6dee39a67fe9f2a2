// test_shim_sor.cpp -- the statistical outlier removal of the reference-facing shim (include/cloud_merger_shim.hpp):
// statisticalOutlierRemoval() and Context::statistical_outlier[_multi] against the C++ statement of
// pcl::StatisticalOutlierRemoval (tests/sor_oracle.cpp), bit for bit. Without a CUDA device it must refuse (exit 77).
#include <cmath>
#include <cstdio>
#include <cstring>
#include <limits>
#include <vector>

#include "cloud_merger_shim.hpp"

using namespace cloud_merger;

extern "C" {
typedef struct {
  double mean, stddev, threshold, sum, sq_sum;
  int64_t n_valid;
  int32_t too_few;
  int32_t n_kept;
} cmo_sor_stats_t;
int cmo_statistical_outlier(const float* xyzi, int64_t n, int mean_k, double std_mul, int negative, int sqrt_mode,
                            float* dist, uint8_t* keep, cmo_sor_stats_t* st);
}

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

static Cloud make_cloud(size_t n) {  // a ring of returns on the ground plus a few strays and NaN rows
  Cloud c;
  c.points.resize(n);
  for (size_t i = 0; i < n; ++i) {
    PointXYZI& p = c.points[i];
    const double r = 2.0 + 30.0 * urand(), az = 6.283185307179586 * urand();
    p.x = static_cast<float>(r * std::cos(az));
    p.y = static_cast<float>(r * std::sin(az));
    p.z = static_cast<float>(0.05 * urand() + (urand() < 0.01 ? 5.0 * urand() : 0.0));
    p.intensity = static_cast<float>(255.0 * urand());
    if (urand() < 0.01) p.y = std::numeric_limits<float>::quiet_NaN();
  }
  c.width = static_cast<uint32_t>(n); c.height = 1; c.is_dense = false;
  return c;
}

static bool same_bits(float a, float b) { return std::memcmp(&a, &b, 4) == 0; }

// the oracle's survivors of `in`, compared with `got` point by point
static void compare(const Cloud& in, const Cloud& got, int mean_k, double std_mul, bool negative, int sqrt_mode,
                    const char* what) {
  const size_t n = in.points.size();
  std::vector<float> xyzi(4 * n + 4), dist(n + 1);
  std::vector<uint8_t> keep(n + 1);
  for (size_t i = 0; i < n; ++i) {
    xyzi[4 * i] = in.points[i].x; xyzi[4 * i + 1] = in.points[i].y;
    xyzi[4 * i + 2] = in.points[i].z; xyzi[4 * i + 3] = in.points[i].intensity;
  }
  cmo_sor_stats_t st;
  CHECK(cmo_statistical_outlier(xyzi.data(), static_cast<int64_t>(n), mean_k, std_mul, negative ? 1 : 0, sqrt_mode,
                                dist.data(), keep.data(), &st) == 0, "%s: oracle", what);
  size_t k = 0;
  bool same = true;
  for (size_t i = 0; i < n; ++i) {
    if (!keep[i]) continue;
    if (k >= got.points.size()) { same = false; break; }
    const PointXYZI& a = got.points[k++];
    const PointXYZI& b = in.points[i];
    same = same && same_bits(a.x, b.x) && same_bits(a.y, b.y) && same_bits(a.z, b.z) && same_bits(a.intensity, b.intensity);
  }
  CHECK(same && k == got.points.size() && static_cast<int64_t>(k) == st.n_kept, "%s: %zu kept, oracle %d", what,
        got.points.size(), st.n_kept);
  CHECK(st.n_kept > 0 && static_cast<size_t>(st.n_kept) < n, "%s: the case removes something and keeps something", what);
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
  {  // the drop-in function, in place
    Cloud::Ptr p(new Cloud(a));
    statisticalOutlierRemoval(ctx, p, 20, 1.0);
    CHECK(ctx.ok(), "statisticalOutlierRemoval: %s", ctx.last_error().c_str());
    compare(a, *p, 20, 1.0, false, CM_SOR_SQRT_FLOAT, "statisticalOutlierRemoval");
  }
  {  // two clouds in one call, negative, the double sqrt
    std::vector<Cloud> out;
    CHECK(ctx.statistical_outlier_multi({&a, &b}, out, 8, 0.5, true, CM_SOR_SQRT_DOUBLE), "multi: %s",
          ctx.last_error().c_str());
    CHECK(out.size() == 2, "multi: two results");
    if (out.size() == 2) {
      compare(a, out[0], 8, 0.5, true, CM_SOR_SQRT_DOUBLE, "multi cloud 0");
      compare(b, out[1], 8, 0.5, true, CM_SOR_SQRT_DOUBLE, "multi cloud 1");
    }
  }
  {  // the radius filter still runs on the same context afterwards
    Cloud out;
    CHECK(ctx.radius_outlier(a, out, 0.15, 1) && !out.points.empty(), "radius_outlier after: %s", ctx.last_error().c_str());
  }
  if (!g_fail) std::printf("shim sor ok\n");
  return g_fail ? 1 : 0;
}
