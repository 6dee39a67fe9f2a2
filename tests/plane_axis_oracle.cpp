// plane_axis_oracle.cpp -- the C++ statement of pcl::SACSegmentation<PointXYZI> with SAC_RANSAC and the models
// SACMODEL_PLANE, SACMODEL_PERPENDICULAR_PLANE and SACMODEL_PARALLEL_PLANE (TEST INFRASTRUCTURE ONLY). It is built in
// one translation unit with oracle/cm_oracle.cpp, so sampler, model, score, eigen33 and refit are that file's own
// (restated from PCL 1.8.1, Eigen 3.3.4, Boost.Random; see the comment there). What it adds is isModelValid of the two
// axis-constrained models, called by countWithinDistance (invalid: 0 inliers) and selectWithinDistance (invalid: no
// inliers), and computeModel's loop with it:
//  PERPENDICULAR  tests only when eps_angle_ > 0: coeff = (a, b, c, 0).normalized(); getAngle3D((ax, ay, az, 0), coeff) =
//                 acos(clamp(double(v1.normalized().dot(v2.normalized())), -1, 1)) -- coeff is normalized twice --
//                 invalid iff min(angle, pi - angle) > eps_angle_.
//  PARALLEL       tests only when eps_angle_ > 0: setAxis stores (ax, ay, az, 0).normalized(), setEpsAngle sin_angle_ =
//                 fabs(sin(eps_angle_)); invalid iff fabs(axis_.dot((a, b, c, 0).normalized())) > sin_angle_.
// A NaN model passes both (every comparison with NaN is false). acos / sin are this process's libm, as in PCL.
// tests/plane_axis_oracle.py compiles it into a temporary directory.
#include "../oracle/cm_oracle.cpp"

namespace {
inline void normalize4(float* v, int order) {
  const float z = sum4(v[0] * v[0], v[1] * v[1], v[2] * v[2], v[3] * v[3], order);
  if (z > 0.0f) {
    const float nrm = std::sqrt(z);
    for (int a = 0; a < 4; ++a) v[a] = v[a] / nrm;
  }
}

bool plane_model_valid(const float* c, int32_t model, const float* axis, double eps_angle, int order) {
  if (model == 0 || !(eps_angle > 0.0)) return true;
  float m[4] = {c[0], c[1], c[2], 0.0f};
  normalize4(m, order);
  float a[4] = {axis[0], axis[1], axis[2], 0.0f};
  normalize4(a, order);
  if (model == 1) {
    normalize4(m, order);
    double rad = sum4(a[0] * m[0], a[1] * m[1], a[2] * m[2], a[3] * m[3], order);
    if (rad < -1.0) rad = -1.0;
    else if (rad > 1.0) rad = 1.0;
    double angle = std::fabs(std::acos(rad));
    angle = std::min(angle, M_PI - angle);
    return !(angle > eps_angle);
  }
  const double sin_angle = std::fabs(std::sin(eps_angle));
  return !(std::fabs(sum4(a[0] * m[0], a[1] * m[1], a[2] * m[2], a[3] * m[3], order)) > sin_angle);
}
}  // namespace

extern "C" {
/* The whole segment() call with setModelType(model) (0 PLANE, 1 PERPENDICULAR_PLANE, 2 PARALLEL_PLANE), setAxis(axis)
 * and setEpsAngle(eps_angle). out_info: [0] found, [1] iterations, [2] draws taken from the sampler, [3] inlier count of
 * the best RANSAC model, [4..6] its sample, [7] iterations whose model failed isModelValid. coeff_ransac / coeff_out: the
 * RANSAC model and what segment() returns (refined when optimize != 0). out_inliers [n]: the final inlier indices,
 * ascending. Returns their number (0 when no model was found). */
int64_t cmo_plane_ransac_model(const float* xyzi, int64_t n, double threshold, double probability, int32_t max_iterations,
                               int32_t optimize, uint32_t seed, int32_t sum_order, int32_t model, const float* axis,
                               double eps_angle, int32_t* out_info, float* coeff_ransac, float* coeff_out,
                               int32_t* out_inliers) {
  int32_t info[8] = {0, 0, 0, 0, -1, -1, -1, 0};
  auto finish = [&](int64_t k) {
    if (out_info) std::memcpy(out_info, info, sizeof(info));
    return k;
  };
  if (n < 3) return finish(0);
  std::vector<int32_t> shuffled(static_cast<size_t>(n));
  for (int64_t i = 0; i < n; ++i) shuffled[i] = static_cast<int32_t>(i);
  Mt19937 rng(seed);
  int iterations = 0, draws = 0;
  int64_t best = -std::numeric_limits<int>::max();
  double k = 1.0;
  const double log_probability = std::log(1.0 - probability);
  const double one_over_indices = 1.0 / static_cast<double>(n);
  float best_c[4] = {0, 0, 0, 0};
  bool have = false;
  while (iterations < k) {
    int32_t sel[3];
    bool got = false;
    for (int check = 0; check < 1000 && !got; ++check) {
      for (int64_t i = 0; i < 3; ++i) {
        const int32_t r = static_cast<int32_t>(rng.next() >> 1);
        std::swap(shuffled[i], shuffled[i + static_cast<int64_t>(static_cast<uint64_t>(r) % static_cast<uint64_t>(n - i))]);
      }
      ++draws;
      sel[0] = shuffled[0]; sel[1] = shuffled[1]; sel[2] = shuffled[2];
      got = plane_sample_good(xyzi + 4 * static_cast<int64_t>(sel[0]), xyzi + 4 * static_cast<int64_t>(sel[1]),
                              xyzi + 4 * static_cast<int64_t>(sel[2]));
    }
    if (!got) break;
    float c[4];
    plane_from_sample(xyzi + 4 * static_cast<int64_t>(sel[0]), xyzi + 4 * static_cast<int64_t>(sel[1]),
                      xyzi + 4 * static_cast<int64_t>(sel[2]), sum_order, c);
    int64_t cnt = 0;
    const bool valid = plane_model_valid(c, model, axis, eps_angle, sum_order);
    if (!valid) ++info[7];  // an iteration with 0 inliers (countWithinDistance), not a skipped sample
    for (int64_t i = 0; valid && i < n; ++i)
      if (plane_distance(c, xyzi + 4 * i, sum_order) < threshold) ++cnt;
    if (cnt > best) {
      best = cnt;
      have = true;
      std::memcpy(best_c, c, sizeof(c));
      info[3] = static_cast<int32_t>(cnt);
      info[4] = sel[0]; info[5] = sel[1]; info[6] = sel[2];
      const double w = static_cast<double>(best) * one_over_indices;
      double p_no_outliers = 1.0 - std::pow(w, 3.0);
      p_no_outliers = std::max(std::numeric_limits<double>::epsilon(), p_no_outliers);
      p_no_outliers = std::min(1.0 - std::numeric_limits<double>::epsilon(), p_no_outliers);
      k = log_probability / std::log(p_no_outliers);
    }
    ++iterations;
    if (iterations > max_iterations) break;
  }
  info[1] = iterations;
  info[2] = draws;
  if (!have) return finish(0);
  info[0] = 1;
  if (coeff_ransac) std::memcpy(coeff_ransac, best_c, sizeof(best_c));
  std::vector<int32_t> inl;
  auto select = [&](const float* c) {
    inl.clear();
    if (!plane_model_valid(c, model, axis, eps_angle, sum_order)) return;
    for (int64_t i = 0; i < n; ++i)
      if (plane_distance(c, xyzi + 4 * i, sum_order) < threshold) inl.push_back(static_cast<int32_t>(i));
  };
  select(best_c);
  float fin_c[4];
  std::memcpy(fin_c, best_c, sizeof(fin_c));
  if (optimize) {
    if (inl.size() >= 4) {
      float acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
      for (int32_t i : inl) {
        const float* p = xyzi + 4 * static_cast<int64_t>(i);
        acc[0] += p[0] * p[0];
        acc[1] += p[0] * p[1];
        acc[2] += p[0] * p[2];
        acc[3] += p[1] * p[1];
        acc[4] += p[1] * p[2];
        acc[5] += p[2] * p[2];
        acc[6] += p[0];
        acc[7] += p[1];
        acc[8] += p[2];
      }
      const float cnt = static_cast<float>(inl.size());
      for (int a = 0; a < 9; ++a) acc[a] = acc[a] / cnt;
      float cov[3][3];
      cov[0][0] = acc[0] - acc[6] * acc[6];
      cov[0][1] = acc[1] - acc[6] * acc[7];
      cov[0][2] = acc[2] - acc[6] * acc[8];
      cov[1][1] = acc[3] - acc[7] * acc[7];
      cov[1][2] = acc[4] - acc[7] * acc[8];
      cov[2][2] = acc[5] - acc[8] * acc[8];
      cov[1][0] = cov[0][1]; cov[2][0] = cov[0][2]; cov[2][1] = cov[1][2];
      float v[3];
      smallest_eigenvector(cov, v);
      fin_c[0] = v[0]; fin_c[1] = v[1]; fin_c[2] = v[2];
      fin_c[3] = -1.0f * sum4(v[0] * acc[6], v[1] * acc[7], v[2] * acc[8], 0.0f * 1.0f, sum_order);
    }
    select(fin_c);
  }
  if (coeff_out) std::memcpy(coeff_out, fin_c, sizeof(fin_c));
  if (out_inliers) std::memcpy(out_inliers, inl.data(), inl.size() * sizeof(int32_t));
  return finish(static_cast<int64_t>(inl.size()));
}

}  // extern "C"
