/*
 * crop_box_oracle.cpp -- CPU oracle of one pcl::CropBox stage (TEST INFRASTRUCTURE ONLY): a restatement of PCL 1.8.1
 * CropBox<PointXYZI>::applyFilter(std::vector<int>&) (filters/impl/crop_box.hpp) that tests/crop_box_oracle.py builds
 * with the flags of oracle/Makefile (-O2 -ffp-contract=off, no -march, no -ffast-math): every float multiply and add
 * rounds on its own, as in PCL's baseline x86-64 build.
 */
#include <algorithm>
#include <cmath>
#include <cstdint>

/* Same layout as cm_crop_box_t of include/cloud_merger_gpu.h. */
typedef struct {
  float min[3], max[3];
  float translation[3];
  float rotation[3];
  float transform[12];
  int32_t negative;
  int32_t reserved;
} cmo_crop_box_t;

/* ---- pcl::CropBox<PointXYZI>::applyFilter(std::vector<int>&) of PCL 1.8.1 (filters/impl/crop_box.hpp) ----------------------
 * Per filter() call PCL derives, in float:
 *   transform = Identity; inverse_transform = Identity;
 *   if (rotation_ != Zero) { getTransformation(0, 0, 0, roll, pitch, yaw, transform); inverse_transform = transform.inverse(); }
 *   transform_matrix_is_identity = transform_.matrix().isIdentity();          // Eigen's fuzzy compare, prec 1e-5
 *   translation_is_zero = (translation_ != Zero);                              // misnamed: true when it is NOT zero
 *   inverse_transform_matrix_is_identity = inverse_transform.matrix().isIdentity();
 * and then per point i (indices_ = every point):
 *   if (!input_->is_dense && !isFinite(point)) continue;                       // removed whatever negative_ is
 *   local = point; if (!transform_matrix_is_identity) local = transformPoint(local, transform_);
 *   if (translation_is_zero) local -= translation_;
 *   if (!inverse_transform_matrix_is_identity) local = transformPoint(local, inverse_transform);
 *   outside = local.x < min.x || local.y < min.y || local.z < min.z || local.x > max.x || local.y > max.y || local.z > max.z;
 *   kept iff (outside == negative_)                                            // a NaN coordinate counts as inside
 * getTransformation (common/impl/eigen.hpp): A = cos(yaw), B = sin(yaw), C = cos(pitch), D = sin(pitch), E = cos(roll),
 * F = sin(roll); rows (A*C, A*DF - B*E, B*F + A*DE), (B*C, A*E + B*DF, B*DE - A*F), (-D, C*F, C*E) with DE = D*E, DF = D*F.
 * Transform::inverse() for Affine: linear = Eigen's 3x3 cofactor inverse, translation = (-linear) * (0, 0, 0) (signed zeros).
 * transformPoint: ((m00*x + m01*y) + m02*z) + m03 per row, the three steps one after another. */
namespace {
inline bool near_identity(const float m[3][4]) {
  const float prec = 1e-5f;  // Eigen::NumTraits<float>::dummy_precision()
  for (int j = 0; j < 4; ++j)      // column by column, as MatrixBase::isIdentity walks it
    for (int i = 0; i < 3; ++i) {
      const float v = m[i][j];
      if (i == j) {
        if (!(std::fabs(v - 1.0f) <= std::min(std::fabs(v), 1.0f) * prec)) return false;  // isApprox(v, 1)
      } else if (!(std::fabs(v) <= std::fabs(1.0f) * prec)) {                               // isMuchSmallerThan(v, 1)
        return false;
      }
    }
  return true;  // row 3 of an Affine3f is exactly 0 0 0 1
}

inline void transform_point(const float m[3][4], float& x, float& y, float& z) {
  const float nx = ((m[0][0] * x + m[0][1] * y) + m[0][2] * z) + m[0][3];
  const float ny = ((m[1][0] * x + m[1][1] * y) + m[1][2] * z) + m[1][3];
  const float nz = ((m[2][0] * x + m[2][1] * y) + m[2][2] * z) + m[2][3];
  x = nx; y = ny; z = nz;
}

inline float cofactor3(const float m[3][4], int i, int j) {
  const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
  return m[i1][j1] * m[i2][j2] - m[i1][j2] * m[i2][j1];
}
}  // namespace

/* The stage on a cloud of n xyzi points whose is_dense flag is given: writes the indices (into the input) of the kept
 * points in input order; returns how many. is_dense == 0 removes non-finite x, y, z first, whatever `negative` is. */
extern "C" int64_t cmo_crop_box(const float* xyzi, int64_t n, int32_t is_dense, const cmo_crop_box_t* box, int32_t* out_idx) {
  float transform[3][4], inverse[3][4] = {{1.f, 0.f, 0.f, 0.f}, {0.f, 1.f, 0.f, 0.f}, {0.f, 0.f, 1.f, 0.f}};
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 4; ++c) transform[r][c] = box->transform[r * 4 + c];
  const float* rot = box->rotation;
  if (rot[0] != 0.f || rot[1] != 0.f || rot[2] != 0.f) {
    const float roll = rot[0], pitch = rot[1], yaw = rot[2];
    const float A = std::cos(yaw), B = std::sin(yaw), C = std::cos(pitch), D = std::sin(pitch), E = std::cos(roll),
                F = std::sin(roll), DE = D * E, DF = D * F;
    const float t[3][4] = {{A * C, A * DF - B * E, B * F + A * DE, 0.f},
                           {B * C, A * E + B * DF, B * DE - A * F, 0.f},
                           {-D, C * F, C * E, 0.f}};
    const float c0 = cofactor3(t, 0, 0), c1 = cofactor3(t, 1, 0), c2 = cofactor3(t, 2, 0);
    const float det = (c0 * t[0][0] + c1 * t[1][0]) + c2 * t[2][0];
    const float invdet = 1.0f / det;
    inverse[0][0] = c0 * invdet; inverse[0][1] = c1 * invdet; inverse[0][2] = c2 * invdet;
    inverse[1][0] = cofactor3(t, 0, 1) * invdet; inverse[1][1] = cofactor3(t, 1, 1) * invdet; inverse[1][2] = cofactor3(t, 2, 1) * invdet;
    inverse[2][0] = cofactor3(t, 0, 2) * invdet; inverse[2][1] = cofactor3(t, 1, 2) * invdet; inverse[2][2] = cofactor3(t, 2, 2) * invdet;
    const float tx = t[0][3], ty = t[1][3], tz = t[2][3];
    for (int r = 0; r < 3; ++r) inverse[r][3] = ((-inverse[r][0]) * tx + (-inverse[r][1]) * ty) + (-inverse[r][2]) * tz;
  }
  const bool apply_transform = !near_identity(transform);
  const float* tr = box->translation;
  const bool apply_translation = tr[0] != 0.f || tr[1] != 0.f || tr[2] != 0.f;
  const bool apply_inverse = !near_identity(inverse);
  int64_t k = 0;
  for (int64_t i = 0; i < n; ++i) {
    float x = xyzi[i * 4 + 0], y = xyzi[i * 4 + 1], z = xyzi[i * 4 + 2];
    if (!is_dense && !(std::isfinite(x) && std::isfinite(y) && std::isfinite(z))) continue;
    if (apply_transform) transform_point(transform, x, y, z);
    if (apply_translation) { x -= tr[0]; y -= tr[1]; z -= tr[2]; }
    if (apply_inverse) transform_point(inverse, x, y, z);
    const bool outside = (x < box->min[0] || y < box->min[1] || z < box->min[2]) ||
                         (x > box->max[0] || y > box->max[1] || z > box->max[2]);
    if (outside == (box->negative != 0)) out_idx[k++] = static_cast<int32_t>(i);
  }
  return k;
}
