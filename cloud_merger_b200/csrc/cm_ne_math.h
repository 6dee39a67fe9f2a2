// cm_ne_math.h -- the per-point arithmetic of pcl::NormalEstimation (PCL 1.8.1) as one statement for the device and the
// host: the kernels of cm_normals.cu, the C++ statement of the tests and (through it) their numpy statement all call these
// functions, so they cannot drift apart. Plain C++ when no CUDA compiler is involved.
//
// Every float operation is rounded on its own (no FMA: __fmul_rn / __fadd_rn / ... on the device; host code including this
// header is built with -ffp-contract=off). The transcendental functions are the one thing PCL takes from the host libm
// (std::atan2 / std::cos / std::sin on floats in computeRoots), and no two libms agree on them (DESIGN section 8), so this
// header fixes a rule of its own: the double-precision functions below, evaluated with IEEE double operations only and
// rounded to float once. They are accurate to a few double ulps, so the float result is the correctly rounded one except
// where the exact value lies within ~2^-50 (relative) of a float midpoint.
#pragma once

#include <stdint.h>
#include <string.h>

#include <cmath>

#ifdef __CUDACC__
#define CM_NE_HD __host__ __device__ __forceinline__
#else
#define CM_NE_HD inline
#endif

namespace cm_ne {

#if defined(__CUDA_ARCH__)
CM_NE_HD double dmul(double a, double b) { return __dmul_rn(a, b); }
CM_NE_HD double dadd(double a, double b) { return __dadd_rn(a, b); }
CM_NE_HD double dsub(double a, double b) { return __dsub_rn(a, b); }
CM_NE_HD double ddiv(double a, double b) { return __ddiv_rn(a, b); }
CM_NE_HD float fmul(float a, float b) { return __fmul_rn(a, b); }
CM_NE_HD float fadd(float a, float b) { return __fadd_rn(a, b); }
CM_NE_HD float fsub(float a, float b) { return __fsub_rn(a, b); }
CM_NE_HD float fdiv(float a, float b) { return __fdiv_rn(a, b); }
CM_NE_HD float fsqrt(float a) { return __fsqrt_rn(a); }
CM_NE_HD uint32_t fbits(float f) { return __float_as_uint(f); }
CM_NE_HD float bitsf(uint32_t u) { return __uint_as_float(u); }
#else
CM_NE_HD double dmul(double a, double b) { return a * b; }
CM_NE_HD double dadd(double a, double b) { return a + b; }
CM_NE_HD double dsub(double a, double b) { return a - b; }
CM_NE_HD double ddiv(double a, double b) { return a / b; }
CM_NE_HD float fmul(float a, float b) { return a * b; }
CM_NE_HD float fadd(float a, float b) { return a + b; }
CM_NE_HD float fsub(float a, float b) { return a - b; }
CM_NE_HD float fdiv(float a, float b) { return a / b; }
CM_NE_HD float fsqrt(float a) { return std::sqrt(a); }
CM_NE_HD uint32_t fbits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
CM_NE_HD float bitsf(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
#endif

constexpr uint32_t QNAN_BITS = 0x7fc00000u;  // std::numeric_limits<float>::quiet_NaN()
CM_NE_HD bool is_nan(float v) { return (fbits(v) & 0x7fffffffu) > 0x7f800000u; }
CM_NE_HD bool is_finite(float v) { return (fbits(v) & 0x7f800000u) != 0x7f800000u; }
CM_NE_HD double dabs(double v) { return v < 0.0 ? -v : v; }
CM_NE_HD float fabs_(float v) { return bitsf(fbits(v) & 0x7fffffffu); }

// ---- the trigonometric rule ---------------------------------------------------------------------------------------------
// sin and cos of a float theta with |theta| <= 1.25 (computeRoots only forms theta in [-fl(pi)/3, fl(pi)/3]): Taylor
// polynomials through x^23 / x^24 in Horner form. Odd / even exactly, signed zeros kept; NaN in, NaN out.
CM_NE_HD float sin_rule(float theta) {
  if (theta == 0.0f) return theta;  // x + x * (x2 * p) would turn -0 into +0
  const double x = theta, x2 = dmul(x, x);
  double p = -3.868170170630684e-23;
  p = dadd(1.9572941063391263e-20, dmul(x2, p));
  p = dadd(-8.22063524662433e-18, dmul(x2, p));
  p = dadd(2.8114572543455206e-15, dmul(x2, p));
  p = dadd(-7.647163731819816e-13, dmul(x2, p));
  p = dadd(1.6059043836821613e-10, dmul(x2, p));
  p = dadd(-2.505210838544172e-08, dmul(x2, p));
  p = dadd(2.7557319223985893e-06, dmul(x2, p));
  p = dadd(-0.0001984126984126984, dmul(x2, p));
  p = dadd(0.008333333333333333, dmul(x2, p));
  p = dadd(-0.16666666666666666, dmul(x2, p));
  return (float)dadd(x, dmul(x, dmul(x2, p)));
}

CM_NE_HD float cos_rule(float theta) {
  const double x = theta, x2 = dmul(x, x);
  double p = 1.6117375710961184e-24;
  p = dadd(-8.896791392450574e-22, dmul(x2, p));
  p = dadd(4.110317623312165e-19, dmul(x2, p));
  p = dadd(-1.5619206968586225e-16, dmul(x2, p));
  p = dadd(4.779477332387385e-14, dmul(x2, p));
  p = dadd(-1.1470745597729725e-11, dmul(x2, p));
  p = dadd(2.08767569878681e-09, dmul(x2, p));
  p = dadd(-2.755731922398589e-07, dmul(x2, p));
  p = dadd(2.48015873015873e-05, dmul(x2, p));
  p = dadd(-0.001388888888888889, dmul(x2, p));
  p = dadd(0.041666666666666664, dmul(x2, p));
  p = dadd(-0.5, dmul(x2, p));
  return (float)dadd(1.0, dmul(x2, p));
}

// atan(t) for 0 <= t <= 1: atan(t) = atan(k/8) + atan(u), u = (t - k/8) / (1 + t k/8), |u| <= 1/16, atan(u) through u^17
CM_NE_HD double atan01(double t) {
  const int k = (int)dadd(dmul(t, 8.0), 0.5);
  // atan(k / 8), selected without an indexed table (which would live in local memory on the device)
  const double a_k = k < 4 ? (k < 2 ? (k == 0 ? 0.0 : 0x1.fd5ba9aac2f6ep-4) : (k == 2 ? 0x1.f5b75f92c80ddp-3 : 0x1.6f61941e4def1p-2))
                           : k < 6 ? (k == 4 ? 0x1.dac670561bb4fp-2 : 0x1.1e00babdefeb4p-1)
                                   : (k == 6 ? 0x1.4978fa3269ee1p-1 : (k == 7 ? 0x1.700a7c5784634p-1 : 0x1.921fb54442d18p-1));
  const double c = dmul((double)k, 0.125);
  const double u = ddiv(dsub(t, c), dadd(1.0, dmul(t, c))), u2 = dmul(u, u);
  double p = 0.058823529411764705;
  p = dadd(-0.06666666666666667, dmul(u2, p));
  p = dadd(0.07692307692307693, dmul(u2, p));
  p = dadd(-0.09090909090909091, dmul(u2, p));
  p = dadd(0.1111111111111111, dmul(u2, p));
  p = dadd(-0.14285714285714285, dmul(u2, p));
  p = dadd(0.2, dmul(u2, p));
  p = dadd(-0.3333333333333333, dmul(u2, p));
  return dadd(a_k, dadd(u, dmul(u, dmul(u2, p))));
}

// atan2 of two floats, with IEEE 754's special values (signed zeros, infinities, NaN) and one rounding to float
CM_NE_HD float atan2_rule(float y, float x) {
  constexpr double PI_HI = 0x1.921fb54442d18p+1, PI_LO = 0x1.1a62633145c07p-53;
  constexpr double PI2_HI = 0x1.921fb54442d18p+0, PI2_LO = 0x1.1a62633145c07p-54;
  if (is_nan(x) || is_nan(y)) return bitsf(QNAN_BITS);
  const bool neg_y = (fbits(y) >> 31) != 0u, neg_x = (fbits(x) >> 31) != 0u;
  const float ax = fabs_(x), ay = fabs_(y);
  const float INF = bitsf(0x7f800000u);
  double r;
  if (ay == 0.0f) r = neg_x ? PI_HI : 0.0;                  // atan2(+-0, -0 or x < 0) = +-pi, else +-0
  else if (ax == 0.0f) r = PI2_HI;                          // y != 0: +-pi/2
  else if (ay == INF) r = ax == INF ? (neg_x ? 0x1.2d97c7f3321d2p+1 : 0x1.921fb54442d18p-1) : PI2_HI;
  else if (ax == INF) r = neg_x ? PI_HI : 0.0;
  else {
    const double dx = ax, dy = ay;
    r = dy <= dx ? atan01(ddiv(dy, dx)) : dadd(dsub(PI2_HI, atan01(ddiv(dx, dy))), PI2_LO);
    if (neg_x) r = dadd(dsub(PI_HI, r), PI_LO);
  }
  const float f = (float)r;
  return neg_y ? -f : f;
}

// ---- PCL 1.8.1 common/impl/eigen.hpp and common/impl/centroid.hpp, float ----------------------------------------------
// Which branches a solve took (the tests check that every case reaches the one it was built for).
enum : uint32_t {
  PATH_ROOTS2 = 1u,       // |c0| < FLT_EPSILON: computeRoots2 straight away
  PATH_TRIG = 2u,         // the closed form with atan2 / cos / sin
  PATH_Q_CLAMP = 4u,      // q > 0 was clamped to +0 (then sqrt(-q) = -0)
  PATH_ROOT0_NEG = 8u,    // roots[0] <= 0 after the closed form: computeRoots2 after all
  PATH_PICK1 = 16u,       // eigen33 took row0 x row1
  PATH_PICK2 = 32u,       //              row0 x row2
  PATH_PICK3 = 64u,       //              row1 x row2
  PATH_NAN_COV = 128u,    // a non-finite covariance entry (documented deviation: quiet NaN x4)
  PATH_FLIP = 256u,       // flipNormalTowardsViewpoint flipped the normal
};

// computeRoots2: roots of x^2 - b x + c, the zero root in front. b * b is a float product; 4.0 * c and the difference
// are double (the literal 4.0), narrowed to float.
CM_NE_HD void roots2(float b, float c, float* roots) {
  roots[0] = 0.0f;
  float d = (float)dsub((double)fmul(b, b), dmul(4.0, (double)c));
  if (d < 0.0f) d = 0.0f;
  const float sd = fsqrt(d);
  roots[2] = fmul(0.5f, fadd(b, sd));
  roots[1] = fmul(0.5f, fsub(b, sd));
}

// computeRoots of the symmetric matrix m = xx xy xz yy yz zz; ascending roots. LIBM: the std:: float functions of the
// host libm instead of the rule (host only; the tests compare the two).
template <bool LIBM>
CM_NE_HD void roots3(const float* m, float* roots, uint32_t* path) {
  const float xx = m[0], xy = m[1], xz = m[2], yy = m[3], yz = m[4], zz = m[5];
  const float c0 = fsub(fsub(fsub(fadd(fmul(fmul(xx, yy), zz), fmul(fmul(fmul(2.0f, xy), xz), yz)), fmul(fmul(xx, yz), yz)),
                             fmul(fmul(yy, xz), xz)),
                        fmul(fmul(zz, xy), xy));
  const float c1 = fsub(fadd(fsub(fadd(fsub(fmul(xx, yy), fmul(xy, xy)), fmul(xx, zz)), fmul(xz, xz)), fmul(yy, zz)),
                        fmul(yz, yz));
  const float c2 = fadd(fadd(xx, yy), zz);
  if (fabs_(c0) < 1.1920928955078125e-7f) {  // Eigen::NumTraits<float>::epsilon()
    *path |= PATH_ROOTS2;
    roots2(c2, c1, roots);
    return;
  }
  *path |= PATH_TRIG;
  const float inv3 = (float)(1.0 / 3.0), sqrt3 = fsqrt(3.0f);
  const float c2_3 = fmul(c2, inv3);
  float a_3 = fmul(fsub(c1, fmul(c2, c2_3)), inv3);
  if (a_3 > 0.0f) a_3 = 0.0f;
  const float half_b = fmul(0.5f, fadd(c0, fmul(c2_3, fsub(fmul(fmul(2.0f, c2_3), c2_3), c1))));
  float q = fadd(fmul(half_b, half_b), fmul(fmul(a_3, a_3), a_3));
  if (q > 0.0f) { q = 0.0f; *path |= PATH_Q_CLAMP; }
  const float rho = fsqrt(-a_3);
  float theta, ct, st;
  if constexpr (LIBM) {
#if !defined(__CUDA_ARCH__)
    theta = fmul(std::atan2(fsqrt(-q), half_b), inv3);
    ct = std::cos(theta);
    st = std::sin(theta);
#endif
  } else {
    theta = fmul(atan2_rule(fsqrt(-q), half_b), inv3);
    ct = cos_rule(theta);
    st = sin_rule(theta);
  }
  roots[0] = fadd(c2_3, fmul(fmul(2.0f, rho), ct));
  roots[1] = fsub(c2_3, fmul(rho, fadd(ct, fmul(sqrt3, st))));
  roots[2] = fsub(c2_3, fmul(rho, fsub(ct, fmul(sqrt3, st))));
  float t;
  if (roots[0] >= roots[1]) { t = roots[0]; roots[0] = roots[1]; roots[1] = t; }
  if (roots[1] >= roots[2]) {
    t = roots[1]; roots[1] = roots[2]; roots[2] = t;
    if (roots[0] >= roots[1]) { t = roots[0]; roots[0] = roots[1]; roots[1] = t; }
  }
  if (roots[0] <= 0.0f) {
    *path |= PATH_ROOT0_NEG;
    roots2(c2, c1, roots);
  }
}

// Eigen 3.3's sum of a 3-vector (squaredNorm): redux_novec_unroller halves the range, a0 + (a1 + a2)
CM_NE_HD float sum3(float a0, float a1, float a2) { return fadd(a0, fadd(a1, a2)); }

CM_NE_HD void cross(const float* u, const float* v, float* o) {
  o[0] = fsub(fmul(u[1], v[2]), fmul(u[2], v[1]));
  o[1] = fsub(fmul(u[2], v[0]), fmul(u[0], v[2]));
  o[2] = fsub(fmul(u[0], v[1]), fmul(u[1], v[0]));
}

// The normal of one neighbourhood from its nine running sums (xx xy xz yy yz zz x y z, PCL's list order) and count:
// computeMeanAndCovarianceMatrix, solvePlaneParameters (pcl::eigen33, the curvature), flipNormalTowardsViewpoint towards
// vp from the query point p. out = nx ny nz curvature, every NaN written as quiet_NaN; roots_out (optional) = the scaled
// matrix's ascending roots. Returns the PATH_* bits.
template <bool LIBM>
CM_NE_HD uint32_t solve(const float* sums, uint32_t count, const float* p, const float* vp, float* out,
                        float* roots_out = nullptr) {
  uint32_t path = 0;
  const float cnt = (float)count;
  float m[9];
  for (int i = 0; i < 9; ++i) m[i] = fdiv(sums[i], cnt);
  float cov[6] = {fsub(m[0], fmul(m[6], m[6])), fsub(m[1], fmul(m[6], m[7])), fsub(m[2], fmul(m[6], m[8])),
                  fsub(m[3], fmul(m[7], m[7])), fsub(m[4], fmul(m[7], m[8])), fsub(m[5], fmul(m[8], m[8]))};
  bool finite = true;
  for (int i = 0; i < 6; ++i) finite = finite && is_finite(cov[i]);
  if (!finite) {
    for (int i = 0; i < 4; ++i) out[i] = bitsf(QNAN_BITS);
    return PATH_NAN_COV;
  }
  // pcl::eigen33(mat, eigenvalue, eigenvector)
  float scale = 0.0f;
  for (int i = 0; i < 6; ++i) scale = fabs_(cov[i]) > scale ? fabs_(cov[i]) : scale;
  if (scale <= 1.17549435e-38f) scale = 1.0f;  // std::numeric_limits<float>::min()
  float s[6];
  for (int i = 0; i < 6; ++i) s[i] = fdiv(cov[i], scale);
  float roots[3];
  roots3<LIBM>(s, roots, &path);
  const float eigenvalue = fmul(roots[0], scale);
  if (roots_out) { roots_out[0] = roots[0]; roots_out[1] = roots[1]; roots_out[2] = roots[2]; }
  const float r0[3] = {fsub(s[0], roots[0]), s[1], s[2]};
  const float r1[3] = {s[1], fsub(s[3], roots[0]), s[4]};
  const float r2[3] = {s[2], s[4], fsub(s[5], roots[0])};
  float v1[3], v2[3], v3[3];
  cross(r0, r1, v1);
  cross(r0, r2, v2);
  cross(r1, r2, v3);
  const float l1 = sum3(fmul(v1[0], v1[0]), fmul(v1[1], v1[1]), fmul(v1[2], v1[2]));
  const float l2 = sum3(fmul(v2[0], v2[0]), fmul(v2[1], v2[1]), fmul(v2[2], v2[2]));
  const float l3 = sum3(fmul(v3[0], v3[0]), fmul(v3[1], v3[1]), fmul(v3[2], v3[2]));
  float v[3], len;
  if (l1 >= l2 && l1 >= l3) { v[0] = v1[0]; v[1] = v1[1]; v[2] = v1[2]; len = l1; path |= PATH_PICK1; }
  else if (l2 >= l1 && l2 >= l3) { v[0] = v2[0]; v[1] = v2[1]; v[2] = v2[2]; len = l2; path |= PATH_PICK2; }
  else { v[0] = v3[0]; v[1] = v3[1]; v[2] = v3[2]; len = l3; path |= PATH_PICK3; }
  const float nrm = fsqrt(len);
  float n[3] = {fdiv(v[0], nrm), fdiv(v[1], nrm), fdiv(v[2], nrm)};
  const float eig_sum = fadd(fadd(cov[0], cov[3]), cov[5]);
  const float curvature = eig_sum != 0.0f ? fabs_(fdiv(eigenvalue, eig_sum)) : 0.0f;
  // flipNormalTowardsViewpoint, the float& overload (features/normal_3d.h): a scalar expression,
  // cos_theta = (vp_x * nx + vp_y * ny + vp_z * nz), evaluated left to right -- not Eigen's dot
  const float dx = fsub(vp[0], p[0]), dy = fsub(vp[1], p[1]), dz = fsub(vp[2], p[2]);
  const float cos_theta = fadd(fadd(fmul(dx, n[0]), fmul(dy, n[1])), fmul(dz, n[2]));
  if (cos_theta < 0.0f) {
    for (int i = 0; i < 3; ++i) n[i] = fmul(n[i], -1.0f);
    path |= PATH_FLIP;
  }
  out[0] = n[0]; out[1] = n[1]; out[2] = n[2]; out[3] = curvature;
  for (int i = 0; i < 4; ++i)
    if (is_nan(out[i])) out[i] = bitsf(QNAN_BITS);
  return path;
}

// one neighbour's contribution to running sum c (0..8): xx xy xz yy yz zz as products, x y z times 1 (exact)
CM_NE_HD float sum_term(int c, float x, float y, float z) {
  const float a = c < 3 ? x : (c < 5 ? y : (c == 5 ? z : (c == 6 ? x : (c == 7 ? y : z))));
  const float b = c >= 6 ? 1.0f : (c == 0 ? x : (c == 1 || c == 3 ? y : z));
  return fmul(a, b);
}

}  // namespace cm_ne
