// ransac_oracle.cpp — CPU ORACLE of PointCloudSensor::fillGroundPlane, a library of its own beside libs3d_oracle.so (loaded by
// oracle/ransac.py; TEST INFRASTRUCTURE, PARITY UNPINNED — see the header of s3d_oracle.cpp).  Built like s3d_oracle.cpp:
// g++ -O2 -std=c++17 -ffp-contract=off -fno-fast-math, so float expressions keep their written, unfused order.
//
// Restates, from the published algorithm (PCL 1.14):
//   slam3d glue   slam3d/sensor/pcl/PointCloudSensor.cpp:362-388 (fillGroundPlane)
//   PCL           pcl/sample_consensus/impl/ransac.hpp          RandomSampleConsensus::computeModel
//                 pcl/sample_consensus/sac_model.h / .hpp       SampleConsensusModel(cloud, random = false), getSamples,
//                                                               drawIndexSample, rnd
//                 pcl/sample_consensus/impl/sac_model_plane.hpp isSampleGood, computeModelCoefficients, countWithinDistance,
//                                                               selectWithinDistance
//   Eigen         Hyperplane::projection, AngleAxis::toRotationMatrix
//
// Definitions (each one is applied by the CUDA path, slam3d_b200/csrc/ransac_math.h, too):
//   * model set-up: the RNG is boost::mt19937 seeded with 12345u (random = false); indices_ = 0..N-1, non-finite points
//     included; shuffled_indices_ = indices_; max_sample_checks_ = 1000; sample size 3;
//   * rnd() = variate_generator<mt19937&, uniform_int<>(0, INT_MAX)>: with a 32-bit engine boost's generate_uniform_int is
//     mt() >> 1 (bucket size 2, never rejected); std::mt19937 gives boost::mt19937's stream;
//   * drawIndexSample: for i = 0, 1, 2: swap(shuffled[i], shuffled[i + rnd() % (N - i)]); the sample is shuffled[0..2] and
//     the permutation carries over to the next draw;
//   * getSamples: up to 1000 draws until isSampleGood accepts; none accepted: empty selection, and the loop ends (failure
//     unless a model was found before).  N < 3 fails at once;
//   * collinearity (isSampleGood and computeModelCoefficients): d = (p1-p0)/(p2-p0) per component in float, good unless
//     d0 == d1 && d2 == d1.  This is the test of PCL <= 1.11; later PCL versions test the norm of the cross product.  The two
//     only disagree on (nearly) degenerate triples.  NaN ratios make a sample good;
//   * coefficients: float cross product of p1-p0 and p2-p0; the 4-vector (n, 0) divided by sqrtf of its left-to-right squared
//     norm when that norm is > 0 (Eigen >= 3.3 normalize(); a zero vector stays zero); d = -(((a x0 + b y0) + c z0) + 0 * 1);
//   * distance |((a x + b y) + c z) + d| in float, left to right, no contraction; a point is an inlier iff its distance,
//     promoted to double, is < threshold (strict).  NaN points are never inliers;
//   * computeModel (threads_ < 0, sequential): k = DBL_MAX; while (iterations_ < k && skipped < 10 max_iterations): rejected
//     coefficients skip++ without iterations_++; a model replaces the best one only with a strictly greater count, then
//     w = count * (1 / N), p = clamp(1 - pow(w, 3), eps, 1 - eps), k = log(1 - probability) / log(p); iterations_++ and
//     break if iterations_ > max_iterations.  fillGroundPlane: threshold 0.01, max_iterations 10000, probability 0.99;
//   * ring fill in double (ScalarType): normal = (double)coeff[0..2] (not renormalised), offset = coeff[3];
//     two_pi = 2 * 3.141592654, step = res / radius; for (ring = res; ring <= radius; ring += res):
//     on_plane = p - ((n0 ring + n1 0) + n2 0 + offset) n with p = (ring, 0, 0); for (angle = 0; angle < two_pi; angle += step):
//     q = AngleAxis(angle, n).toRotationMatrix() * on_plane with Eigen's formula (sin_axis = sin(angle) n, c = cos(angle),
//     cos1_axis = (1 - c) n, off-diagonals tmp -+ sin_axis, diagonal cos1_axis .* n + c), rows left to right; the point is
//     (float)q with w = 1.  sin and cos are libm's.


#include "../include/s3d_b200.h"

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <random>
#include <vector>

namespace {

struct P4 { float x, y, z, w; };

struct RansacOut {
  bool ok = false;
  float coeff[4] = {0, 0, 0, 0};
  int iterations = 0;
  std::vector<uint32_t> inliers;
};

struct RansacPlaneModel {
  const P4* pts;
  std::vector<uint32_t> shuffled;
  std::mt19937 rng{12345u};
  explicit RansacPlaneModel(const P4* p, size_t n) : pts(p), shuffled(n) { for (size_t i = 0; i < n; ++i) shuffled[i] = (uint32_t)i; }

  int rnd() { return (int)(rng() >> 1); }

  void drawIndexSample(uint32_t sample[3]) {
    const size_t n = shuffled.size();
    for (size_t i = 0; i < 3; ++i) std::swap(shuffled[i], shuffled[i + ((size_t)rnd() % (n - i))]);
    for (int i = 0; i < 3; ++i) sample[i] = shuffled[i];
  }

  bool isSampleGood(const uint32_t s[3]) const {
    const P4 &p0 = pts[s[0]], &p1 = pts[s[1]], &p2 = pts[s[2]];
    const float d0 = (p1.x - p0.x) / (p2.x - p0.x);
    const float d1 = (p1.y - p0.y) / (p2.y - p0.y);
    const float d2 = (p1.z - p0.z) / (p2.z - p0.z);
    return !(d0 == d1 && d2 == d1);
  }

  // false: empty selection
  bool getSamples(uint32_t sample[3]) {
    if (shuffled.size() < 3) return false;
    for (int it = 0; it < 1000; ++it) {
      drawIndexSample(sample);
      if (isSampleGood(sample)) return true;
    }
    return false;
  }

  bool computeModelCoefficients(const uint32_t s[3], float c[4]) const {
    if (!isSampleGood(s)) return false;
    const P4 &p0 = pts[s[0]], &p1 = pts[s[1]], &p2 = pts[s[2]];
    const float ax = p1.x - p0.x, ay = p1.y - p0.y, az = p1.z - p0.z;
    const float bx = p2.x - p0.x, by = p2.y - p0.y, bz = p2.z - p0.z;
    c[0] = ay * bz - az * by;
    c[1] = az * bx - ax * bz;
    c[2] = ax * by - ay * bx;
    c[3] = 0.f;
    const float n2 = ((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2]) + c[3] * c[3];
    if (n2 > 0.f) { const float s = std::sqrt(n2); for (int i = 0; i < 4; ++i) c[i] = c[i] / s; }
    c[3] = -(((c[0] * p0.x + c[1] * p0.y) + c[2] * p0.z) + c[3] * 1.0f);
    return true;
  }

  static float distance(const float c[4], const P4& p) { return std::fabs(((c[0] * p.x + c[1] * p.y) + c[2] * p.z) + c[3]); }

  uint64_t countWithinDistance(const float c[4], double threshold) const {
    uint64_t n = 0;
    for (size_t i = 0; i < shuffled.size(); ++i) if ((double)distance(c, pts[i]) < threshold) ++n;
    return n;
  }
};

static RansacOut ransac_plane_fit(const P4* pts, size_t n, double threshold, int max_iterations, double probability) {
  RansacOut out;
  RansacPlaneModel model(pts, n);
  double k = std::numeric_limits<double>::max();
  const double log_probability = std::log(1.0 - probability);
  const double one_over_indices = 1.0 / static_cast<double>(n);
  const unsigned max_skip = (unsigned)max_iterations * 10u;
  unsigned skipped = 0;
  uint64_t best = 0;
  int iterations = 0;
  bool have_model = false;
  while (iterations < k && skipped < max_skip) {
    uint32_t selection[3];
    if (!model.getSamples(selection)) break;
    float c[4];
    if (!model.computeModelCoefficients(selection, c)) { ++skipped; continue; }
    const uint64_t count = model.countWithinDistance(c, threshold);
    if (count > best) {
      best = count;
      std::memcpy(out.coeff, c, sizeof c);
      have_model = true;
      const double w = static_cast<double>(count) * one_over_indices;
      double p_no_outliers = 1.0 - std::pow(w, 3.0);
      p_no_outliers = std::max(std::numeric_limits<double>::epsilon(), p_no_outliers);
      p_no_outliers = std::min(1.0 - std::numeric_limits<double>::epsilon(), p_no_outliers);
      k = log_probability / std::log(p_no_outliers);
    }
    ++iterations;
    if (iterations > max_iterations) break;
  }
  out.iterations = iterations;
  if (!have_model) return out;
  out.ok = true;
  for (size_t i = 0; i < n; ++i) if ((double)RansacPlaneModel::distance(out.coeff, pts[i]) < threshold) out.inliers.push_back((uint32_t)i);
  return out;
}

static void ground_rings(double res, double radius, std::vector<double>& rings, std::vector<double>& angles) {
  const double two_pi = 2 * 3.141592654, step = res / radius;
  for (double ring = res; ring <= radius; ring += res) rings.push_back(ring);
  for (double angle = 0; angle < two_pi; angle += step) angles.push_back(angle);
}

// the points fillGroundPlane appends, ring-major, angle-minor
static void ground_fill(const float coeff[4], double res, double radius, std::vector<P4>& out) {
  const double n[3] = {coeff[0], coeff[1], coeff[2]};
  const double offset = coeff[3];
  std::vector<double> rings, angles;
  ground_rings(res, radius, rings, angles);
  for (double ring : rings) {
    const double p[3] = {ring, 0.0, 0.0};
    const double sd = ((n[0] * p[0] + n[1] * p[1]) + n[2] * p[2]) + offset;
    double v[3];
    for (int i = 0; i < 3; ++i) v[i] = p[i] - sd * n[i];
    for (double angle : angles) {
      const double sa = std::sin(angle), c = std::cos(angle);
      double sin_axis[3], cos1_axis[3], R[3][3];
      for (int i = 0; i < 3; ++i) { sin_axis[i] = sa * n[i]; cos1_axis[i] = (1.0 - c) * n[i]; }
      double tmp = cos1_axis[0] * n[1];
      R[0][1] = tmp - sin_axis[2]; R[1][0] = tmp + sin_axis[2];
      tmp = cos1_axis[0] * n[2];
      R[0][2] = tmp + sin_axis[1]; R[2][0] = tmp - sin_axis[1];
      tmp = cos1_axis[1] * n[2];
      R[1][2] = tmp - sin_axis[0]; R[2][1] = tmp + sin_axis[0];
      for (int i = 0; i < 3; ++i) R[i][i] = cos1_axis[i] * n[i] + c;
      P4 q;
      q.x = (float)((R[0][0] * v[0] + R[0][1] * v[1]) + R[0][2] * v[2]);
      q.y = (float)((R[1][0] * v[0] + R[1][1] * v[1]) + R[1][2] * v[2]);
      q.z = (float)((R[2][0] * v[0] + R[2][1] * v[1]) + R[2][2] * v[2]);
      q.w = 1.f;
      out.push_back(q);
    }
  }
}

}  // namespace

extern "C" {
// pcl::RandomSampleConsensus + SampleConsensusModelPlane as fillGroundPlane runs it.  inliers (may be NULL) holds cloud.n entries.
// Returns S3D_OK, or S3D_INVALID_ARGUMENT when RANSAC finds no model (N < 3 included).
int s3d_oracle_fit_plane_ransac(s3d_cloud cloud, double threshold, int max_iterations, double probability, float coefficients[4],
                                int32_t* iterations, uint64_t* n_inliers, uint32_t* inliers) {
  const RansacOut r = ransac_plane_fit(reinterpret_cast<const P4*>(cloud.xyzw), cloud.n, threshold, max_iterations, probability);
  *iterations = r.iterations;
  *n_inliers = r.inliers.size();
  std::memcpy(coefficients, r.coeff, sizeof r.coeff);
  if (inliers && !r.inliers.empty()) std::memcpy(inliers, r.inliers.data(), 4 * r.inliers.size());
  return r.ok ? S3D_OK : S3D_INVALID_ARGUMENT;
}

// Number of points fillGroundPlane appends for (map_resolution, radius).
uint64_t s3d_oracle_ground_fill_size(double map_resolution, double radius) {
  std::vector<double> rings, angles;
  ground_rings(map_resolution, radius, rings, angles);
  return (uint64_t)rings.size() * angles.size();
}

// fillGroundPlane: RANSAC (threshold 0.01, PCL defaults), then the rings; out_xyzw holds s3d_oracle_ground_fill_size() points.
int s3d_oracle_fill_ground_plane(s3d_cloud cloud, double map_resolution, double radius, float* out_xyzw, uint64_t* n_out, float coefficients[4]) {
  const RansacOut r = ransac_plane_fit(reinterpret_cast<const P4*>(cloud.xyzw), cloud.n, 0.01, 10000, 0.99);
  *n_out = 0;
  if (!r.ok) return S3D_INVALID_ARGUMENT;
  if (coefficients) std::memcpy(coefficients, r.coeff, sizeof r.coeff);
  std::vector<P4> pts;
  ground_fill(r.coeff, map_resolution, radius, pts);
  if (!pts.empty()) std::memcpy(out_xyzw, pts.data(), pts.size() * sizeof(P4));
  *n_out = pts.size();
  return S3D_OK;
}

// Test hook: the first n outputs of mt19937 seeded with `seed` (mt_out) and of rnd() on a second engine with the same seed.
void s3d_oracle_test_rng(uint32_t seed, int n, uint32_t* mt_out, int32_t* rnd_out) {
  std::mt19937 a(seed);
  for (int i = 0; i < n; ++i) mt_out[i] = a();
  RansacPlaneModel m(nullptr, 0);
  m.rng.seed(seed);
  for (int i = 0; i < n; ++i) rnd_out[i] = m.rnd();
}
}  // extern "C"
