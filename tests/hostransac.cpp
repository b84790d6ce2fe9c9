// Host build of slam3d_b200/csrc/ransac_math.h for the CPU test-suite (tests/test_hostransac.py).
// Test-only: runs the GPU path's pieces on the host in the GPU path's order — the sampler emits blocks of B planes, every plane
// is counted against every point with ransac_distance(), RansacReplay consumes the counts in loop order — and the ring fill with
// ground_fill_lists() / ground_fill_point().  Built with -ffp-contract=off.
#include <cuda_runtime.h>  // float4 and make_float4 on the host

#include <cstring>
#include <vector>

#include "../slam3d_b200/csrc/ransac_math.h"

using namespace s3d;

extern "C" {

// Returns 0 and the fit, or 6 when no model was found; *blocks receives the number of blocks run.
int hr_fit(const float* xyzw, uint32_t n, double threshold, int max_iterations, double probability, int B, float coeff[4], int32_t* iterations,
           uint64_t* n_inliers, uint32_t* inliers, int32_t* blocks) {
  const float4* pts = reinterpret_cast<const float4*>(xyzw);
  *iterations = 0; *n_inliers = 0; *blocks = 0;
  if (n < 3) return 6;
  std::vector<uint32_t> shuffled(n);
  for (uint32_t i = 0; i < n; ++i) shuffled[i] = i;
  std::vector<uint32_t> mt(kMtWords);
  int32_t mti = 0;
  mt_seed(mt.data(), mti, kRansacSeed);
  bool ended = false;
  const float t = ransac_float_threshold(threshold);
  RansacReplay R(n, max_iterations, probability);
  while (R.wants_more()) {
    const int count = (int)std::min<uint64_t>((uint64_t)B, R.remaining_bound());
    std::vector<float4> planes(count);
    std::vector<int> flags(count);
    uint32_t s[3] = {shuffled[0], shuffled[1], shuffled[2]};
    for (int b = 0; b < count; ++b) {
      uint32_t sel[3];
      float4 plane = make_float4(NAN, NAN, NAN, NAN);
      flags[b] = ended ? kRansacNoSample : ransac_next_hypothesis(mt.data(), mti, shuffled.data(), s, n, pts, &plane, sel);
      if (flags[b] == kRansacNoSample) ended = true;
      planes[b] = flags[b] == kRansacScored ? plane : make_float4(NAN, NAN, NAN, NAN);
    }
    shuffled[0] = s[0]; shuffled[1] = s[1]; shuffled[2] = s[2];
    ++*blocks;
    for (int b = 0; b < count && R.wants_more(); ++b) {
      uint64_t c = 0;
      for (uint32_t i = 0; i < n; ++i) c += ransac_distance(planes[b], pts[i].x, pts[i].y, pts[i].z) < t ? 1 : 0;
      const float p[4] = {planes[b].x, planes[b].y, planes[b].z, planes[b].w};
      R.consume(flags[b], c, p);
    }
  }
  *iterations = R.iterations;
  if (!R.have_model) return 6;
  std::memcpy(coeff, R.best, sizeof R.best);
  const float4 m = make_float4(R.best[0], R.best[1], R.best[2], R.best[3]);
  uint64_t k = 0;
  for (uint32_t i = 0; i < n; ++i)
    if (ransac_distance(m, pts[i].x, pts[i].y, pts[i].z) < t) { if (inliers) inliers[k] = i; ++k; }
  *n_inliers = k;
  return 0;
}

// fill points for the plane coeff; out holds ground_fill size points.  Returns 0, or 6 on bad arguments.
int hr_fill(const float coeff[4], double res, double radius, float* out, uint64_t* n_out) {
  std::vector<double> rings, sin_a, cos_a;
  if (!ground_fill_lists(res, radius, (1ull << 31) - 1, &rings, &sin_a, &cos_a, n_out)) return 6;
  const double n[3] = {coeff[0], coeff[1], coeff[2]};
  float4* o = reinterpret_cast<float4*>(out);
  for (size_t i = 0; i < rings.size(); ++i)
    for (size_t j = 0; j < sin_a.size(); ++j) o[i * sin_a.size() + j] = ground_fill_point(n, (double)coeff[3], rings[i], sin_a[j], cos_a[j]);
  return 0;
}

// the first n outputs of mt_next() after mt_seed(seed)
void hr_mt(uint32_t seed, int n, uint32_t* out) {
  std::vector<uint32_t> mt(kMtWords);
  int32_t mti = 0;
  mt_seed(mt.data(), mti, seed);
  for (int i = 0; i < n; ++i) out[i] = mt_next(mt.data(), mti);
}

}  // extern "C"
