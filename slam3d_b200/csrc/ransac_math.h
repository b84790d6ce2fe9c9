// ransac_math.h — the arithmetic of PointCloudSensor::fillGroundPlane (slam3d/sensor/pcl/PointCloudSensor.cpp:362-388), callable
// from host and device.
//
// pcl::RandomSampleConsensus with pcl::SampleConsensusModelPlane (definitions: DESIGN.md 6f), split so that
// the GPU can run ahead of PCL's sequential loop (DESIGN.md 6f):
//   * the sampler (getSamples / drawIndexSample / isSampleGood / computeModelCoefficients) depends on the points and on the seeded
//     RNG only, never on inlier counts: ransac_next_hypothesis() emits the next iteration's plane and runs on one GPU thread;
//   * counting is the hot path: ransac_distance() per (point, plane), in ransac.cu;
//   * RansacReplay applies the loop's acceptance / k / skipped / max_iterations rules to the counts in loop order, on the host;
//   * the ring fill: ground_fill_lists() builds the loops' ring and angle values on the host, ground_fill_point() forms one point.
// Float and double operations go through the *_rn helpers on the device, so nvcc cannot contract them; the host build (the
// oracle's compiler flags, -ffp-contract=off) keeps the written order too.
#pragma once

#include <stdint.h>

#include <cfloat>
#include <cmath>
#include <limits>
#include <vector>

#if defined(__CUDACC__)
#define S3D_RS_HD __host__ __device__ __forceinline__
#else
#define S3D_RS_HD inline
#endif

namespace s3d {

constexpr int kMtWords = 624;
constexpr uint32_t kRansacSeed = 12345u;     // SampleConsensusModel(cloud, random = false)
constexpr int kRansacMaxSampleChecks = 1000; // max_sample_checks_
enum RansacFlag { kRansacScored = 0, kRansacSkipped = 1, kRansacNoSample = 2 };

S3D_RS_HD float rs_mul(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fmul_rn(a, b);
#else
  return a * b;
#endif
}
S3D_RS_HD float rs_add(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fadd_rn(a, b);
#else
  return a + b;
#endif
}
S3D_RS_HD float rs_sub(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fsub_rn(a, b);
#else
  return a - b;
#endif
}
S3D_RS_HD float rs_div(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fdiv_rn(a, b);
#else
  return a / b;
#endif
}
S3D_RS_HD float rs_sqrt(float a) {
#if defined(__CUDA_ARCH__)
  return __fsqrt_rn(a);
#else
  return std::sqrt(a);
#endif
}
S3D_RS_HD double rs_dmul(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
S3D_RS_HD double rs_dadd(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}
S3D_RS_HD double rs_dsub(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dsub_rn(a, b);
#else
  return a - b;
#endif
}

// ---- MT19937 (boost::mt19937 == std::mt19937) ---------------------------------------------------------------------------
S3D_RS_HD void mt_seed(uint32_t* mt, int32_t& mti, uint32_t seed) {
  mt[0] = seed;
  for (int i = 1; i < kMtWords; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
  mti = kMtWords;
}

S3D_RS_HD uint32_t mt_next(uint32_t* mt, int32_t& mti) {
  if (mti >= kMtWords) {
    for (int i = 0; i < kMtWords; ++i) {
      const uint32_t y = (mt[i] & 0x80000000u) | (mt[i + 1 < kMtWords ? i + 1 : 0] & 0x7FFFFFFFu);
      mt[i] = mt[i + 397 < kMtWords ? i + 397 : i + 397 - kMtWords] ^ (y >> 1) ^ ((y & 1u) ? 0x9908B0DFu : 0u);
    }
    mti = 0;
  }
  uint32_t y = mt[mti++];
  y ^= y >> 11;
  y ^= (y << 7) & 0x9D2C5680u;
  y ^= (y << 15) & 0xEFC60000u;
  y ^= y >> 18;
  return y;
}

// rnd(): variate_generator<mt19937&, uniform_int<>(0, INT_MAX)>; boost's generate_uniform_int reduces it to mt() >> 1.
S3D_RS_HD uint32_t ransac_rnd(uint32_t* mt, int32_t& mti) { return mt_next(mt, mti) >> 1; }

// ---- plane model -----------------------------------------------------------------------------------------------------------
// isSampleGood / the collinearity test of computeModelCoefficients: dy1dy2 = (p1-p0)/(p2-p0) per component, good unless
// dy1dy2[0] == dy1dy2[1] && dy1dy2[2] == dy1dy2[1] (PCL's ratio test; NaN ratios make a sample "good").
S3D_RS_HD bool ransac_sample_good(float4 p0, float4 p1, float4 p2) {
  const float d0 = rs_div(rs_sub(p1.x, p0.x), rs_sub(p2.x, p0.x));
  const float d1 = rs_div(rs_sub(p1.y, p0.y), rs_sub(p2.y, p0.y));
  const float d2 = rs_div(rs_sub(p1.z, p0.z), rs_sub(p2.z, p0.z));
  return !(d0 == d1 && d2 == d1);
}

// computeModelCoefficients after the collinearity test: float cross product of p1-p0 and p2-p0, 4-vector (n, 0) normalised by
// sqrtf of its left-to-right squared norm (Eigen >= 3.3 normalize(): a zero vector stays zero), then d = -(n . (p0, 1)).
S3D_RS_HD float4 ransac_plane(float4 p0, float4 p1, float4 p2) {
  const float ax = rs_sub(p1.x, p0.x), ay = rs_sub(p1.y, p0.y), az = rs_sub(p1.z, p0.z);
  const float bx = rs_sub(p2.x, p0.x), by = rs_sub(p2.y, p0.y), bz = rs_sub(p2.z, p0.z);
  float a = rs_sub(rs_mul(ay, bz), rs_mul(az, by));
  float b = rs_sub(rs_mul(az, bx), rs_mul(ax, bz));
  float c = rs_sub(rs_mul(ax, by), rs_mul(ay, bx));
  const float n2 = rs_add(rs_add(rs_add(rs_mul(a, a), rs_mul(b, b)), rs_mul(c, c)), rs_mul(0.f, 0.f));
  if (n2 > 0.f) {
    const float s = rs_sqrt(n2);
    a = rs_div(a, s); b = rs_div(b, s); c = rs_div(c, s);
  }
  const float dot = rs_add(rs_add(rs_add(rs_mul(a, p0.x), rs_mul(b, p0.y)), rs_mul(c, p0.z)), rs_mul(0.f, 1.f));
  return make_float4(a, b, c, -dot);
}

// countWithinDistance / selectWithinDistance: |((a x + b y) + c z) + d| in float; a point counts iff it is < threshold
S3D_RS_HD float ransac_distance(float4 m, float x, float y, float z) {
  return fabsf(rs_add(rs_add(rs_add(rs_mul(m.x, x), rs_mul(m.y, y)), rs_mul(m.z, z)), m.w));
}

// One iteration's getSamples + computeModelCoefficients.  shuffled: the persistent permutation (shuffled_indices_, n entries);
// s: its first three entries, which the caller keeps in registers and writes back when it stops.  pts: the n points.
// Returns the flag; the plane and the sample go to *plane / sel.
S3D_RS_HD int ransac_next_hypothesis(uint32_t* mt, int32_t& mti, uint32_t* shuffled, uint32_t (&s)[3], uint32_t n, const float4* pts,
                                     float4* plane, uint32_t (&sel)[3]) {
  for (int check = 0; check < kRansacMaxSampleChecks; ++check) {
    // drawIndexSample: swap(shuffled[i], shuffled[i + rnd() % (n - i)]) for i = 0, 1, 2
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < 3; ++i) {
      const uint32_t j = (uint32_t)i + ransac_rnd(mt, mti) % (n - (uint32_t)i);
      const uint32_t t = s[i];
      if (j == 1) { s[i] = s[1]; s[1] = t; }
      else if (j == 2) { s[i] = s[2]; s[2] = t; }
      else if (j >= 3) { s[i] = shuffled[j]; shuffled[j] = t; }
    }
    const float4 p0 = pts[s[0]], p1 = pts[s[1]], p2 = pts[s[2]];
    if (!ransac_sample_good(p0, p1, p2)) continue;
    sel[0] = s[0]; sel[1] = s[1]; sel[2] = s[2];
    if (!ransac_sample_good(p0, p1, p2)) return kRansacSkipped;  // computeModelCoefficients repeats the test
    *plane = ransac_plane(p0, p1, p2);
    return kRansacScored;
  }
  return kRansacNoSample;
}

// ---- host side of the loop ---------------------------------------------------------------------------------------------------
// Double-precision float threshold test: for a float distance d, (double)d < threshold  <=>  d < ransac_float_threshold(threshold).
inline float ransac_float_threshold(double threshold) {
  float t = (float)threshold;
  if ((double)t < threshold) t = std::nextafter(t, INFINITY);
  return t;
}

// RandomSampleConsensus::computeModel (threads_ < 0), fed one iteration at a time in loop order.
struct RansacReplay {
  double k = DBL_MAX;
  double log_probability = 0, one_over_indices = 0;
  int32_t iterations = 0;
  uint32_t skipped = 0, max_skip = 0;
  int32_t max_iterations = 0;
  uint64_t best_count = 0;
  float best[4] = {0, 0, 0, 0};
  bool have_model = false, ended = false;

  RansacReplay(uint64_t n, int max_it, double probability)
      : log_probability(std::log(1.0 - probability)), one_over_indices(1.0 / (double)n), max_skip((uint32_t)max_it * 10u),
        max_iterations(max_it) {}
  // the while condition, checked before each getSamples
  bool wants_more() const { return !ended && (double)iterations < k && skipped < max_skip; }
  // upper bound of the iterations still to come (at least 1 while the loop runs): a block of this many is never wasted
  uint64_t remaining_bound() const {
    const double lim = std::fmin(k, (double)max_iterations + 1.0);
    const double r = std::ceil(lim) - (double)iterations;
    return r < 1.0 ? 1 : (uint64_t)r;
  }
  void consume(int flag, uint64_t count, const float plane[4]) {
    if (flag == kRansacNoSample) { ended = true; return; }
    if (flag == kRansacSkipped) { ++skipped; return; }
    if (count > best_count) {
      best_count = count;
      for (int i = 0; i < 4; ++i) best[i] = plane[i];
      have_model = true;
      const double w = (double)count * one_over_indices;
      double p_no_outliers = 1.0 - std::pow(w, 3.0);
      p_no_outliers = std::fmax(std::numeric_limits<double>::epsilon(), p_no_outliers);
      p_no_outliers = std::fmin(1.0 - std::numeric_limits<double>::epsilon(), p_no_outliers);
      k = log_probability / std::log(p_no_outliers);
    }
    ++iterations;
    if (iterations > max_iterations) ended = true;
  }
};

// fillGroundPlane's loops: for (ring = res; ring <= radius; ring += res), for (angle = 0; angle < 2 * 3.141592654; angle += res / radius),
// both accumulated in double.  sin/cos of every angle with libm, once.  false when the fill would exceed max_points.
inline bool ground_fill_lists(double res, double radius, uint64_t max_points, std::vector<double>* rings, std::vector<double>* sin_a,
                              std::vector<double>* cos_a, uint64_t* n_points) {
  const double two_pi = 2 * 3.141592654, step = res / radius;
  uint64_t nr = 0, na = 0;
  for (double ring = res; ring <= radius; ring += res) {
    if (++nr > max_points) return false;
    if (rings) rings->push_back(ring);
  }
  for (double angle = 0; angle < two_pi; angle += step) {
    if (++na > max_points) return false;
    if (sin_a) { sin_a->push_back(std::sin(angle)); cos_a->push_back(std::cos(angle)); }
  }
  if (nr && na > max_points / nr) return false;
  *n_points = nr * na;
  return true;
}

// One fill point: on_plane = p - (n . p + offset) n with p = (ring, 0, 0) (Hyperplane::projection), then
// AngleAxis(angle, n).toRotationMatrix() * on_plane (Eigen's formula, rows left to right), cast to float.
S3D_RS_HD float4 ground_fill_point(const double n[3], double offset, double ring, double sa, double ca) {
  const double sd = rs_dadd(rs_dadd(rs_dadd(rs_dmul(n[0], ring), rs_dmul(n[1], 0.0)), rs_dmul(n[2], 0.0)), offset);
  const double v0 = rs_dsub(ring, rs_dmul(sd, n[0])), v1 = rs_dsub(0.0, rs_dmul(sd, n[1])), v2 = rs_dsub(0.0, rs_dmul(sd, n[2]));
  const double s0 = rs_dmul(sa, n[0]), s1 = rs_dmul(sa, n[1]), s2 = rs_dmul(sa, n[2]);
  const double om = rs_dsub(1.0, ca);
  const double c0 = rs_dmul(om, n[0]), c1 = rs_dmul(om, n[1]), c2 = rs_dmul(om, n[2]);
  double R[3][3];
  double tmp = rs_dmul(c0, n[1]);
  R[0][1] = rs_dsub(tmp, s2); R[1][0] = rs_dadd(tmp, s2);
  tmp = rs_dmul(c0, n[2]);
  R[0][2] = rs_dadd(tmp, s1); R[2][0] = rs_dsub(tmp, s1);
  tmp = rs_dmul(c1, n[2]);
  R[1][2] = rs_dsub(tmp, s0); R[2][1] = rs_dadd(tmp, s0);
  R[0][0] = rs_dadd(rs_dmul(c0, n[0]), ca); R[1][1] = rs_dadd(rs_dmul(c1, n[1]), ca); R[2][2] = rs_dadd(rs_dmul(c2, n[2]), ca);
  float4 o;
  o.x = (float)rs_dadd(rs_dadd(rs_dmul(R[0][0], v0), rs_dmul(R[0][1], v1)), rs_dmul(R[0][2], v2));
  o.y = (float)rs_dadd(rs_dadd(rs_dmul(R[1][0], v0), rs_dmul(R[1][1], v1)), rs_dmul(R[1][2], v2));
  o.z = (float)rs_dadd(rs_dadd(rs_dmul(R[2][0], v0), rs_dmul(R[2][1], v1)), rs_dmul(R[2][2], v2));
  o.w = 1.0f;
  return o;
}

}  // namespace s3d
