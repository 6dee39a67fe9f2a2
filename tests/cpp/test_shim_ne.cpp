// test_shim_ne.cpp -- the normal estimation of the reference-facing shim (include/cloud_merger_shim.hpp): estimateNormals()
// and Context::normals[_multi] against the C++ statement of pcl::NormalEstimation (tests/ne_oracle.cpp): the same bits.
// Without a CUDA device it must refuse (exit 77).
#include <array>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <limits>
#include <vector>

#include "cloud_merger_shim.hpp"

using namespace cloud_merger;

extern "C" int cmo_normals(const float* xyzi, int64_t n, double radius, const float* vp, int trig_mode, int exhaustive,
                           float* out, int32_t* counts, uint32_t* paths, float* roots);

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

static Cloud make_cloud(size_t n) {  // noisy patches of a ground plane and a wall, duplicates and NaN rows
  Cloud c;
  c.points.resize(n);
  for (size_t i = 0; i < n; ++i) {
    PointXYZI& p = c.points[i];
    const bool wall = urand() < 0.3;
    const double u = 6.0 * urand(), v = 3.0 * urand(), e = 0.02 * urand();
    p.x = static_cast<float>(wall ? 6.0 + e : u);
    p.y = static_cast<float>(wall ? u : v);
    p.z = static_cast<float>(wall ? v : e);
    p.intensity = static_cast<float>(255.0 * urand());
    if (i > 0 && urand() < 0.05) p = c.points[i - 1];
    if (urand() < 0.01) p.y = std::numeric_limits<float>::quiet_NaN();
  }
  c.width = static_cast<uint32_t>(n); c.height = 1; c.is_dense = false;
  return c;
}

static void compare(const Cloud& in, const std::vector<float>& got, double radius, const std::array<float, 3>& vp,
                    const char* what) {
  const size_t n = in.points.size();
  std::vector<float> xyzi(4 * n + 4), want(4 * n + 4);
  for (size_t i = 0; i < n; ++i) {
    xyzi[4 * i] = in.points[i].x; xyzi[4 * i + 1] = in.points[i].y;
    xyzi[4 * i + 2] = in.points[i].z; xyzi[4 * i + 3] = in.points[i].intensity;
  }
  CHECK(cmo_normals(xyzi.data(), static_cast<int64_t>(n), radius, vp.data(), 0, 0, want.data(), nullptr, nullptr,
                    nullptr) == 0, "%s: oracle", what);
  CHECK(got.size() == 4 * n, "%s: %zu floats for %zu points", what, got.size(), n);
  size_t bad = 0, finite = 0;
  for (size_t k = 0; k < got.size() && k < 4 * n; ++k) {
    uint32_t a, b;
    std::memcpy(&a, &got[k], 4);
    std::memcpy(&b, &want[k], 4);
    bad += a != b;
    finite += std::isfinite(got[k]);
  }
  CHECK(bad == 0, "%s: %zu floats differ", what, bad);
  CHECK(finite > 2 * n, "%s: the case has normals", what);
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
  const std::array<float, 3> vp{{3.0f, 1.5f, 1.8f}};
  {  // the drop-in function
    Cloud::Ptr p(new Cloud(a));
    std::vector<float> out;
    estimateNormals(ctx, p, 0.3, vp, out);
    CHECK(ctx.ok(), "estimateNormals: %s", ctx.last_error().c_str());
    compare(a, out, 0.3, vp, "estimateNormals");
  }
  {  // two clouds in one call, the default viewpoint, a radius that is not a float
    std::vector<std::vector<float>> out;
    CHECK(ctx.normals_multi({&a, &b}, out, 0.1), "multi: %s", ctx.last_error().c_str());
    CHECK(out.size() == 2, "multi: two results");
    if (out.size() == 2) {
      compare(a, out[0], 0.1, {{0.f, 0.f, 0.f}}, "multi cloud 0");
      compare(b, out[1], 0.1, {{0.f, 0.f, 0.f}}, "multi cloud 1");
    }
  }
  {  // the radius filter still runs on the same context afterwards
    Cloud out;
    CHECK(ctx.radius_outlier(a, out, 0.15, 1) && !out.points.empty(), "radius_outlier after: %s", ctx.last_error().c_str());
  }
  if (!g_fail) std::printf("shim ne ok\n");
  return g_fail ? 1 : 0;
}
