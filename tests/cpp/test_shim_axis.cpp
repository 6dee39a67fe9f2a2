// test_shim_axis.cpp -- the axis-constrained plane models of the reference-facing shim (include/cloud_merger_shim.hpp):
// Params::sac_model / max_angle / axis through Context::plane_ransac[_multi], removeGround and proceedConfig, against the
// C++ statement of pcl::SACSegmentation (tests/plane_axis_oracle.cpp), bit for bit. Without a CUDA device it must refuse
// (exit 77).
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "cloud_merger_shim.hpp"

using namespace cloud_merger;

extern "C" int64_t cmo_plane_ransac_model(const float* xyzi, int64_t n, double threshold, double probability,
                                          int32_t max_iterations, int32_t optimize, uint32_t seed, int32_t sum_order,
                                          int32_t model, const float* axis, double eps_angle, int32_t* out_info,
                                          float* coeff_ransac, float* coeff_out, int32_t* out_inliers);

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

static uint64_t g_rng = 0x9E3779B97F4A7C15ull;
static double urand() {  // splitmix64
  uint64_t z = (g_rng += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (z >> 11) * (1.0 / 9007199254740992.0);
}

// a zone whose wall (x = 6, facing the sensor) holds more points than its ground (z = -1.8, slightly tilted)
static Cloud wall_zone(size_t n_ground, size_t n_wall, size_t n_clutter) {
  Cloud c;
  for (size_t i = 0; i < n_ground + n_wall + n_clutter; ++i) {
    PointXYZI p;
    const double u = 12.0 * urand() - 6.0, v = 8.0 * urand() - 4.0, e = 0.04 * (urand() - 0.5);
    if (i < n_ground) { p.x = (float)u; p.y = (float)v; p.z = (float)(-1.8 + 0.01 * u + e); }
    else if (i < n_ground + n_wall) { p.x = (float)(6.0 + e); p.y = (float)v; p.z = (float)(-1.7 + 2.0 * urand()); }
    else { p.x = (float)u; p.y = (float)v; p.z = (float)(-1.5 + 1.8 * urand()); }
    p.intensity = (float)(255.0 * urand());
    c.points.push_back(p);
  }
  c.width = static_cast<uint32_t>(c.points.size()); c.height = 1; c.is_dense = true;
  return c;
}

static bool same_bits(float a, float b) { return std::memcmp(&a, &b, 4) == 0; }

// the oracle's segment() + ExtractIndices of `in` with p's settings and eps, against the shim's ground / rest and model
static void compare(const Cloud& in, const Params& p, double eps, const Cloud& ground, const Cloud& rest, const cm_plane_t* m,
                    const char* what) {
  const size_t n = in.points.size();
  std::vector<float> xyzi(4 * n + 4);
  for (size_t i = 0; i < n; ++i) {
    xyzi[4 * i] = in.points[i].x; xyzi[4 * i + 1] = in.points[i].y;
    xyzi[4 * i + 2] = in.points[i].z; xyzi[4 * i + 3] = in.points[i].intensity;
  }
  int32_t info[8];
  float cr[4], co[4];
  std::vector<int32_t> inl(n + 1);
  const int64_t k = cmo_plane_ransac_model(xyzi.data(), static_cast<int64_t>(n), p.distance_threshold, p.prob, p.max_iterations,
                                           1, 12345u, p.sum_order, p.sac_model, p.axis, eps, info, cr, co, inl.data());
  std::vector<char> is_in(n, 0);
  for (int64_t j = 0; j < k; ++j) is_in[static_cast<size_t>(inl[static_cast<size_t>(j)])] = 1;
  size_t gi = 0, ri = 0;
  bool same = true;
  for (size_t i = 0; i < n && same; ++i) {
    const Cloud& c = is_in[i] ? ground : rest;
    size_t& at = is_in[i] ? gi : ri;
    if (at >= c.points.size()) { same = false; break; }
    const PointXYZI& a = c.points[at++];
    const PointXYZI& b = in.points[i];
    same = same_bits(a.x, b.x) && same_bits(a.y, b.y) && same_bits(a.z, b.z) && same_bits(a.intensity, b.intensity);
  }
  CHECK(same && gi == ground.points.size() && ri == rest.points.size() && static_cast<int64_t>(gi) == k,
        "%s: ground %zu / rest %zu, oracle %lld inliers", what, ground.points.size(), rest.points.size(), (long long)k);
  if (m) {
    CHECK(m->found == info[0] && m->iterations == info[1] && m->draws == info[2] && m->best_count == info[3] &&
              m->rejected == info[7], "%s: found %d it %d draws %d best %d rejected %d, oracle %d %d %d %d %d", what, m->found,
          m->iterations, m->draws, m->best_count, m->rejected, info[0], info[1], info[2], info[3], info[7]);
    bool cs = true;
    for (int a = 0; a < 4; ++a) cs = cs && same_bits(m->coeff[a], co[a]) && same_bits(m->coeff_ransac[a], cr[a]);
    CHECK(cs, "%s: coefficients differ from the oracle", what);
  }
}

int main() {
  if (cm_device_count() == 0) {
    std::printf("no CUDA device: the shim has no CPU path (expected on the build box)\n");
    Context ctx(1024);
    CHECK(!ctx.ok(), "Context must fail without a GPU");
    return g_fail ? 1 : 77;  // 77 = skipped
  }
  const double ten_deg = 10.0 * M_PI / 180.0;
  const Cloud zone = wall_zone(700, 1400, 300), other = wall_zone(900, 300, 200);
  Params plane_p;  // the reference's SACMODEL_PLANE: max_angle and axis are ignored
  plane_p.max_angle = ten_deg;
  Params perp_p;
  perp_p.sac_model = CM_SAC_PERPENDICULAR_PLANE;
  perp_p.max_angle = ten_deg;
  Params par_p;
  par_p.sac_model = CM_SAC_PARALLEL_PLANE;
  par_p.max_angle = ten_deg;
  for (const Params* p : {&plane_p, &perp_p, &par_p}) {
    Context ctx(1 << 14, 2, 0, *p);
    CHECK(ctx.ok(), "Context: %s", ctx.last_error().c_str());
    Cloud g, r;
    cm_plane_t m;
    CHECK(ctx.plane_ransac(zone, g, r, &m), "plane_ransac: %s", ctx.last_error().c_str());
    compare(zone, *p, p->max_angle, g, r, &m, "plane_ransac");
    // the wall holds more points: only the perpendicular model finds the ground (normal near z)
    const bool horizontal = std::fabs(m.coeff[2]) > 0.9f;
    CHECK(horizontal == (p->sac_model == CM_SAC_PERPENDICULAR_PLANE), "model %d: normal (%g, %g, %g)", p->sac_model,
          m.coeff[0], m.coeff[1], m.coeff[2]);
    std::vector<Cloud> gs, rs;
    std::vector<cm_plane_t> ms;
    CHECK(ctx.plane_ransac_multi({&zone, &other}, gs, rs, &ms) && gs.size() == 2, "multi: %s", ctx.last_error().c_str());
    if (gs.size() == 2) {
      compare(zone, *p, p->max_angle, gs[0], rs[0], &ms[0], "multi cloud 0");
      compare(other, *p, p->max_angle, gs[1], rs[1], &ms[1], "multi cloud 1");
    }
    // removeGround: its max_angle argument is the eps_angle (float, widened); the RANSAC runs on the lower z window
    const float z_lo = -2.5f, z_hi = 0.0f, max_angle = static_cast<float>(0.2);
    std::vector<cm_zone_t> zones(1);
    zones[0].n_pass = 1; zones[0].pass[0] = cm_pass_t{2, z_lo, z_hi, 0};
    std::vector<Cloud> low;
    CHECK(ctx.zone_split(zone, zones, low) && low.size() == 1, "zone_split: %s", ctx.last_error().c_str());
    Cloud::Ptr in(new Cloud(zone)), ng(new Cloud), gr(new Cloud);
    removeGround(ctx, in, ng, gr, z_lo, z_hi, max_angle);
    CHECK(ctx.ok(), "removeGround: %s", ctx.last_error().c_str());
    if (low.size() == 1) {
      Cloud g2, r2;
      CHECK(ctx.plane_ransac(low[0], g2, r2, planeConfig(*p, static_cast<double>(max_angle))), "plane on the window");
      compare(low[0], *p, static_cast<double>(max_angle), *gr, r2, nullptr, "removeGround");
    }
    // proceedConfig carries the model, the axis and max_angle into the one-call zone pass
    const cm_proceed_cfg_t cfg = proceedConfig(*p, {ZonePart{12.0f, -6.0f, 2.5f}}, {});
    CHECK(cfg.plane.model == p->sac_model && cfg.plane.eps_angle == p->max_angle && cfg.plane.axis[2] == 1.0f &&
              cfg.plane.axis[0] == 0.0f && cfg.plane.axis[1] == 0.0f, "proceedConfig: plane settings");
  }
  if (!g_fail) std::printf("shim axis ok\n");
  return g_fail ? 1 : 0;
}
