// ne_oracle.cpp -- C++ statement of pcl::NormalEstimation<PointXYZI, Normal>::computeFeature (PCL 1.8.1) with a radius
// search (TEST INFRASTRUCTURE ONLY). For every query: the finite points p with fl((dx*dx + dy*dy) + dz*dz) < r2,
// r2 = (float)(radius * radius), the query itself included, sorted with std::sort on (d2, index) -- FLANN's
// RadiusResultSet order -- then the nine running sums in that order and cm_ne_math.h's solve (the code the kernels run),
// with the trig rule (trig_mode 0) or the host libm's std::atan2 / std::cos / std::sin on floats (trig_mode 1).
// The neighbours are collected exhaustively (exhaustive = 1) or from a grid of cells 1.01 radius wide in double (a superset
// of the points within the float bound, filtered by the same float test); the tests check that the two agree.
// Also the checks of the trig rule against correctly rounded references and the host libm.
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <random>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../cloud_merger_b200/csrc/cm_ne_math.h"

namespace {

bool finite3(const float* p) { return std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]); }

float d2_of(const float* q, const float* p) {
  const float ex = q[0] - p[0], ey = q[1] - p[1], ez = q[2] - p[2];
  return (ex * ex + ey * ey) + ez * ez;
}

int g_threads = 0;  // 0: one per hardware thread (at most 16)

template <typename F>
void parallel_for(int64_t n, F f) {
  const int T = g_threads > 0 ? g_threads : (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
  std::vector<std::thread> th;
  std::atomic<int64_t> next(0);
  for (int t = 0; t < T; ++t)
    th.emplace_back([&]() {
      for (;;) {
        const int64_t b = next.fetch_add(4096);
        if (b >= n) return;
        for (int64_t i = b; i < std::min(n, b + 4096); ++i) f(i);
      }
    });
  for (auto& x : th) x.join();
}

uint32_t fb(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
float bf(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }

// the correctly rounded float of a double reference value r (accurate to a few ulps): false when r lies within 2^-46
// (relative) of a float midpoint and the long double value long_ref() lies within 2^-60 of it as well
template <typename L>
bool cr_float(double r, L long_ref, float* out) {
  const float f = (float)r;
  if (!std::isfinite(f) || r == 0.0) { *out = f; return true; }
  const float g = nextafterf(f, (double)f < r ? INFINITY : -INFINITY);
  const double mid = ((double)f + (double)g) * 0.5;
  if (fabs(r - mid) > ldexp(fabs(r), -46)) { *out = f; return true; }
  const long double ml = ((long double)f + (long double)g) * 0.5L, rl = long_ref();
  if (fabsl(rl - ml) > ldexpl(fabsl(rl), -60)) { *out = (rl < ml) == ((long double)f < ml) ? f : g; return true; }
  return false;
}

}  // namespace

extern "C" {

// threads of the statement (1: the one-core CPU baseline of the benchmark); 0 restores the default
void cmo_set_threads(int n) { g_threads = n; }

// normals of one cloud: out [n][4] nx ny nz curvature, counts [n] neighbourhood sizes (0 for non-finite queries),
// paths [n] the PATH_* bits, roots [n][3] the scaled matrix's roots (NaN where no solve ran); the last three may be NULL
int cmo_normals(const float* xyzi, int64_t n, double radius, const float* vp, int trig_mode, int exhaustive, float* out,
                int32_t* counts, uint32_t* paths, float* roots) {
  const float r2 = (float)(radius * radius);
  const double cell = radius * 1.01;
  std::unordered_map<uint64_t, std::vector<int64_t>> grid;
  auto cell_of = [&](const float* p, int64_t* c) {
    for (int a = 0; a < 3; ++a) c[a] = (int64_t)floor((double)p[a] / cell);
  };
  auto hkey = [](int64_t x, int64_t y, int64_t z) {
    return ((uint64_t)(x & 0x1FFFFF) << 42) | ((uint64_t)(y & 0x1FFFFF) << 21) | (uint64_t)(z & 0x1FFFFF);
  };
  if (!exhaustive)
    for (int64_t i = 0; i < n; ++i)
      if (finite3(xyzi + 4 * i)) {
        int64_t c[3];
        cell_of(xyzi + 4 * i, c);
        grid[hkey(c[0], c[1], c[2])].push_back(i);
      }
  const float nanf_ = bf(cm_ne::QNAN_BITS);
  parallel_for(n, [&](int64_t i) {
    const float* q = xyzi + 4 * i;
    float* o = out + 4 * i;
    for (int k = 0; k < 4; ++k) o[k] = nanf_;
    if (counts) counts[i] = 0;
    if (paths) paths[i] = 0;
    if (roots) for (int k = 0; k < 3; ++k) roots[3 * i + k] = nanf_;
    if (!finite3(q)) return;
    std::vector<std::pair<float, int64_t>> nb;
    auto test = [&](int64_t j) {
      const float* p = xyzi + 4 * j;
      if (!finite3(p)) return;
      const float d = d2_of(q, p);
      if (d < r2) nb.emplace_back(d, j);
    };
    if (exhaustive) {
      for (int64_t j = 0; j < n; ++j) test(j);
    } else {
      int64_t c[3];
      cell_of(q, c);
      for (int64_t dz = -1; dz <= 1; ++dz)
        for (int64_t dy = -1; dy <= 1; ++dy)
          for (int64_t dx = -1; dx <= 1; ++dx) {
            auto it = grid.find(hkey(c[0] + dx, c[1] + dy, c[2] + dz));
            if (it == grid.end()) continue;
            for (int64_t j : it->second) test(j);
          }
    }
    std::sort(nb.begin(), nb.end());  // FLANN: (distance, index)
    if (counts) counts[i] = (int32_t)nb.size();
    if (nb.size() < 3) return;
    float sums[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (const auto& e : nb) {
      const float* p = xyzi + 4 * e.second;
      for (int k = 0; k < 9; ++k) sums[k] += cm_ne::sum_term(k, p[0], p[1], p[2]);
    }
    uint32_t path;
    float* ro = roots ? roots + 3 * i : nullptr;
    if (trig_mode == 1) path = cm_ne::solve<true>(sums, (uint32_t)nb.size(), q, vp, o, ro);
    else path = cm_ne::solve<false>(sums, (uint32_t)nb.size(), q, vp, o, ro);
    if (paths) paths[i] = path;
  });
  return 0;
}

// the solve of given sums (the numpy statement's route to the shared code): n rows of 9 sums, counts, query points
int cmo_solve(const float* sums, const int64_t* counts, const float* xyzi, int64_t n, const float* vp, int trig_mode,
              float* out, uint32_t* paths) {
  for (int64_t i = 0; i < n; ++i) {
    float* o = out + 4 * i;
    const float* q = xyzi + 4 * i;
    if (!finite3(q) || counts[i] < 3) {
      for (int k = 0; k < 4; ++k) o[k] = bf(cm_ne::QNAN_BITS);
      if (paths) paths[i] = 0;
      continue;
    }
    const uint32_t p = trig_mode == 1 ? cm_ne::solve<true>(sums + 9 * i, (uint32_t)counts[i], q, vp, o)
                                      : cm_ne::solve<false>(sums + 9 * i, (uint32_t)counts[i], q, vp, o);
    if (paths) paths[i] = p;
  }
  return 0;
}

float cmo_atan2(float y, float x) { return cm_ne::atan2_rule(y, x); }
float cmo_cos(float x) { return cm_ne::cos_rule(x); }
float cmo_sin(float x) { return cm_ne::sin_rule(x); }

// Every float theta with bits in [lo, hi]: the rule's sin / cos against the correctly rounded float (glibc's double
// function, and long double near a midpoint). st[0] floats, [1] sin mismatches, [2] cos mismatches, [3] unresolved
// (within 2^-60 of a midpoint even in long double: either float accepted), [4] sinf == rule, [5] cosf == rule,
// [6] sign symmetry failures on the negated theta (every 64th)
int cmo_sincos_check(uint32_t lo, uint32_t hi, int64_t* st) {
  std::atomic<int64_t> a[7];
  for (auto& v : a) v = 0;
  const int64_t n = (int64_t)hi - lo + 1;
  parallel_for((n + 1023) / 1024, [&](int64_t blk) {
    int64_t s[7] = {0, 0, 0, 0, 0, 0, 0};
    for (int64_t k = blk * 1024; k < std::min(n, blk * 1024 + 1024); ++k) {
      const float x = bf(lo + (uint32_t)k);
      const float gs = cm_ne::sin_rule(x), gc = cm_ne::cos_rule(x);
      float ws, wc;
      ++s[0];
      if (cr_float(sin((double)x), [&] { return sinl((long double)x); }, &ws)) { if (fb(ws) != fb(gs)) ++s[1]; } else ++s[3];
      if (cr_float(cos((double)x), [&] { return cosl((long double)x); }, &wc)) { if (fb(wc) != fb(gc)) ++s[2]; } else ++s[3];
      if (sinf(x) == gs) ++s[4];
      if (cosf(x) == gc) ++s[5];
      if ((k & 63) == 0 && (fb(cm_ne::sin_rule(-x)) != (fb(gs) ^ 0x80000000u) || fb(cm_ne::cos_rule(-x)) != fb(gc))) ++s[6];
    }
    for (int j = 0; j < 7; ++j) a[j] += s[j];
  });
  for (int j = 0; j < 7; ++j) st[j] = a[j];
  return 0;
}

// n sampled (y, x) pairs: half random finite bit patterns (y of either sign), half uniform in y in [0, 1], x in [-1, 1].
// st[0] samples, [1] mismatches against the correctly rounded float of atan2l, [2] unresolved, [3] atan2f == rule
int cmo_atan2_check(uint64_t seed, int64_t n, int64_t* st) {
  std::atomic<int64_t> a[4];
  for (auto& v : a) v = 0;
  const int64_t blocks = (n + 65535) / 65536;
  parallel_for(blocks, [&](int64_t blk) {
    std::mt19937_64 rng(seed * 1000003ull + (uint64_t)blk);
    std::uniform_real_distribution<float> u01(0.0f, 1.0f);
    int64_t s[4] = {0, 0, 0, 0};
    for (int64_t k = blk * 65536; k < std::min(n, blk * 65536 + 65536); ++k) {
      float y, x;
      if (k & 1) {
        do { y = bf((uint32_t)rng()); x = bf((uint32_t)rng()); } while (!std::isfinite(y) || !std::isfinite(x));
      } else {
        y = u01(rng);
        x = 2.0f * u01(rng) - 1.0f;
      }
      const float g = cm_ne::atan2_rule(y, x);
      float w;
      ++s[0];
      const long double rl = atan2l((long double)y, (long double)x);
      if (cr_float((double)rl, [&] { return rl; }, &w)) { if (fb(w) != fb(g)) ++s[1]; } else ++s[2];
      if (fb(atan2f(y, x)) == fb(g)) ++s[3];
    }
    for (int j = 0; j < 4; ++j) a[j] += s[j];
  });
  for (int j = 0; j < 4; ++j) st[j] = a[j];
  return 0;
}

}  // extern "C"
