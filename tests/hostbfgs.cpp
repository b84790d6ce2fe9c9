// Host build of the BFGS state machine of slam3d_b200/csrc/gicp_bfgs.h for the CPU test-suite (tests/test_hostbfgs.py).
// Test-only: drives the machine that runs on the GPU on explicit correspondences, forming every requested evaluation's sums in
// point order on the host (float residual exactly as PCL forms it; built with -ffp-contract=off), and counts which decisions of
// the line search the cases reach.
#include <cstring>

static long long hb_hit_count[16];
#define S3D_BFGS_HIT(k) (++hb_hit_count[(k)])

#include "../slam3d_b200/csrc/gicp_math.h"

namespace {
// Eigen Matrix4f * Vector4f with w = 1 (same order as common.cuh transform_mv)
inline void transform_mv(const float* T, const float* p, float* o) {
  o[0] = ((T[0] * p[0] + T[4] * p[1]) + T[8] * p[2]) + T[12];
  o[1] = ((T[1] * p[0] + T[5] * p[1]) + T[9] * p[2]) + T[13];
  o[2] = ((T[2] * p[0] + T[6] * p[1]) + T[10] * p[2]) + T[14];
}
// f and gradient at x from the 13 residual sums (+ count) of one evaluation pass, summed in point order
void evaluate(const float* moved, const float* fixed, const double* M6, int m, const double x[6], double& f, double (&g)[6]) {
  float T[16];
  s3d::matrix_from_state(x, T);
  double sums[s3d::kNumMoments];
  for (int i = 0; i < s3d::kNumMoments; ++i) sums[i] = 0.0;
  for (int i = 0; i < m; ++i) {
    const float* p = moved + 4 * i; const float* q = fixed + 4 * i; const double* M = M6 + 6 * i;
    float pp[3];
    transform_mv(T, p, pp);
    const double d[3] = {(double)(pp[0] - q[0]), (double)(pp[1] - q[1]), (double)(pp[2] - q[2])};
    const double Mf[3][3] = {{M[0], M[1], M[2]}, {M[1], M[3], M[4]}, {M[2], M[4], M[5]}};
    const double phi[4] = {p[0], p[1], p[2], 1.0};
    double Md[3];
    for (int a = 0; a < 3; ++a) Md[a] = Mf[a][0] * d[0] + Mf[a][1] * d[1] + Mf[a][2] * d[2];
    for (int a = 0; a < 3; ++a) for (int c = 0; c < 4; ++c) sums[60 + a * 4 + c] += Md[a] * phi[c];
    sums[72] += d[0] * Md[0] + d[1] * Md[1] + d[2] * Md[2];
    sums[73] += 1.0;
  }
  s3d::Euler E;
  s3d::euler_derivs(x, E, false);
  f = sums[72] / sums[73];
  for (int i = 0; i < 6; ++i) g[i] = s3d::objective_entry(sums, E, i);
}
}  // namespace

extern "C" {
// estimateRigidTransformationBFGS through the resumable state machine.  T column-major float in/out (unchanged on failure);
// returns 0, or 2 where PCL throws (fewer than 4 correspondences, or a solve it rejects) — the oracle's test hook's convention.
int hb_bfgs(const float* moved, const float* fixed, const double* M6, int m, float* T, int max_inner, int* inner_done, int* evaluations) {
  *inner_done = 0;
  if (evaluations) *evaluations = 0;
  if (m < 4) return 2;
  s3d::BfgsState st;
  s3d::bfgs_begin(st, T);
  double f, g[6];
  int evals = 1;
  evaluate(moved, fixed, M6, m, st.xc, f, g);
  while (s3d::bfgs_advance(st, f, g, max_inner)) {
    evaluate(moved, fixed, M6, m, st.xc, f, g);
    ++evals;
  }
  *inner_done = st.it;
  if (evaluations) *evaluations = evals;
  if (st.failed) return 2;
  s3d::matrix_from_state(st.x, T);
  return 0;
}
// decision counters of the machine (s3d::BfgsBranch), optionally cleared
int hb_hits(long long* out, int reset) {
  for (int i = 0; i < s3d::kBfgsBranches; ++i) out[i] = hb_hit_count[i];
  if (reset) std::memset(hb_hit_count, 0, sizeof hb_hit_count);
  return s3d::kBfgsBranches;
}
}
