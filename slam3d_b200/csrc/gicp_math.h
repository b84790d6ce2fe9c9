// gicp_math.h — scalar FP64 math of the GICP optimiser, callable from host and device.
//
// What it computes (reference: PCL gicp.hpp as driven by slam3d doICP, PointCloudSensor.cpp:52-82; SURVEY A.3/A.5):
//   * closed 3x3 / 6x6 symmetric eigen-decompositions (cyclic Jacobi) — covariance regularisation and the
//     Newton step of estimateRigidTransformationNewton;
//   * the GICP objective f(x) = 1/m sum d^T M d, d = T(x) p - q, its exact gradient and Hessian in the
//     (t, ZYX-Euler) parametrisation, assembled from 74 sums of one pass over the correspondences, and PCL's inner
//     optimisers as resumable state machines (one yield per objective evaluation): the Newton one of PCL >= 1.14 here, the
//     BFGS one of PCL <= 1.13 in gicp_bfgs.h (included at the end).
//
// B200-first design note: of the 74 sums, 60 (sum M (x) phi phi^T, phi = (p,1)) do not depend on x and give the whole
// Hessian except its second-derivative term; an evaluation pass only adds the 13 sums that contain the residual d.
// d is formed per point exactly as PCL forms it (float32 transform T(x), float subtraction, then double), because
// PCL's line search decisions are dominated by that float rounding once the step is below ~1e-5 m; mirroring it makes
// the GPU follow the oracle's iterate sequence instead of merely converging to a nearby point.
#pragma once

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define S3D_HD __host__ __device__ __forceinline__
#else
#define S3D_HD inline
#endif

namespace s3d {

constexpr int kNumMoments = 74;  // 60 (S) + 12 (v) + 1 (s0) + 1 (count)
constexpr double kGicpEpsilon = 1e-3;  // gicp_epsilon_ (PCL default; not exposed by slam3d)

// index of the unordered pair (a,b), a,b in 0..2  -> 0..5   (00,01,02,11,12,22)
S3D_HD int sym3(int a, int b) { if (a > b) { int t = a; a = b; b = t; } return a == 0 ? b : (a == 1 ? 2 + b : 5); }
// index of the unordered pair (c,e), c,e in 0..3  -> 0..9   (00,01,02,03,11,12,13,22,23,33)
S3D_HD int sym4(int c, int e) { if (c > e) { int t = c; c = e; e = t; } return c == 0 ? e : (c == 1 ? 3 + e : (c == 2 ? 5 + e : 9)); }
// moment layout: S[sym3(a,b)*10 + sym4(c,e)] at 0..59, v[a*4+c] at 60..71, s0 at 72, count at 73

// Cyclic Jacobi for symmetric NxN: A = V diag(w) V^T (A destroyed). Same operation order as the oracle's.
template <int N>
S3D_HD void jacobi_eigen(double (&A)[N][N], double (&V)[N][N], double (&w)[N]) {
  for (int i = 0; i < N; ++i) for (int j = 0; j < N; ++j) V[i][j] = (i == j) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = 0, diag = 0;
    for (int i = 0; i < N; ++i) { diag += A[i][i] * A[i][i]; for (int j = i + 1; j < N; ++j) off += A[i][j] * A[i][j]; }
    if (off <= 1e-34 * diag || off == 0.0) break;
    for (int p = 0; p < N - 1; ++p)
      for (int q = p + 1; q < N; ++q) {
        const double apq = A[p][q];
        if (apq == 0.0) continue;
        const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < N; ++k) { const double akp = A[k][p], akq = A[k][q]; A[k][p] = c * akp - s * akq; A[k][q] = s * akp + c * akq; }
        for (int k = 0; k < N; ++k) { const double apk = A[p][k], aqk = A[q][k]; A[p][k] = c * apk - s * aqk; A[q][k] = s * apk + c * aqk; }
        for (int k = 0; k < N; ++k) { const double vkp = V[k][p], vkq = V[k][q]; V[k][p] = c * vkp - s * vkq; V[k][q] = s * vkp + c * vkq; }
      }
  }
  for (int i = 0; i < N; ++i) w[i] = A[i][i];
}

// GICP covariance regularisation (SURVEY A.3 step 4): from the 3x3 moment covariance, the unit eigenvector of the
// eigenvalue of smallest magnitude (= last singular vector of JacobiSVD).  C_reg = I - (1 - eps) n n^T.
S3D_HD void smallest_eigenvector3(double (&cov)[3][3], double (&n)[3]) {
  double V[3][3], w[3];
  jacobi_eigen<3>(cov, V, w);
  // descending |w| with a stable order, like the oracle's stable_sort; the last one is the normal
  int o0 = 0, o1 = 1, o2 = 2;
  if (fabs(w[o1]) > fabs(w[o0])) { int t = o0; o0 = o1; o1 = t; }
  if (fabs(w[o2]) > fabs(w[o1])) { int t = o1; o1 = o2; o2 = t; }
  if (fabs(w[o1]) > fabs(w[o0])) { int t = o0; o0 = o1; o1 = t; }
  n[0] = V[0][o2]; n[1] = V[1][o2]; n[2] = V[2][o2];
}

struct Euler { double R[3][3]; double dR[3][3][3]; double ddR[3][3][3][3]; };

S3D_HD void mat3_mul(const double (&A)[3][3], const double (&B)[3][3], double (&C)[3][3]) {
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { double s = 0; for (int k = 0; k < 3; ++k) s += A[i][k] * B[k][j]; C[i][j] = s; }
}

S3D_HD void euler_factor(double ang, int axis, double (&R)[3][3], double (&dR)[3][3], double (&ddR)[3][3]) {
  const double c = cos(ang), s = sin(ang);
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) R[i][j] = dR[i][j] = ddR[i][j] = 0.0;
  const int i = (axis + 1) % 3, j = (axis + 2) % 3;
  R[axis][axis] = 1.0;
  R[i][i] = c;  R[i][j] = -s; R[j][i] = s;  R[j][j] = c;
  dR[i][i] = -s; dR[i][j] = -c; dR[j][i] = c;  dR[j][j] = -s;
  ddR[i][i] = -c; ddR[i][j] = s; ddR[j][i] = -s; ddR[j][j] = -c;
}

// R = Rz(x5) Ry(x4) Rx(x3) and its first/second derivatives w.r.t. (x3,x4,x5)   (gicp.hpp applyState / computeRDerivative)
S3D_HD void euler_derivs(const double x[6], Euler& E, bool second) {
  double X[3][3], dX[3][3], ddX[3][3], Y[3][3], dY[3][3], ddY[3][3], Z[3][3], dZ[3][3], ddZ[3][3], ZY[3][3], T[3][3];
  euler_factor(x[3], 0, X, dX, ddX);
  euler_factor(x[4], 1, Y, dY, ddY);
  euler_factor(x[5], 2, Z, dZ, ddZ);
  mat3_mul(Z, Y, ZY);
  mat3_mul(ZY, X, E.R);
  mat3_mul(ZY, dX, E.dR[0]);
  mat3_mul(Z, dY, T); mat3_mul(T, X, E.dR[1]);
  mat3_mul(dZ, Y, T); mat3_mul(T, X, E.dR[2]);
  if (!second) return;
  mat3_mul(ZY, ddX, E.ddR[0][0]);
  mat3_mul(Z, ddY, T); mat3_mul(T, X, E.ddR[1][1]);
  mat3_mul(ddZ, Y, T); mat3_mul(T, X, E.ddR[2][2]);
  mat3_mul(Z, dY, T); mat3_mul(T, dX, E.ddR[0][1]);
  mat3_mul(dZ, Y, T); mat3_mul(T, dX, E.ddR[0][2]);
  mat3_mul(dZ, dY, T); mat3_mul(T, X, E.ddR[1][2]);
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) {
    E.ddR[1][0][i][j] = E.ddR[0][1][i][j]; E.ddR[2][0][i][j] = E.ddR[0][2][i][j]; E.ddR[2][1][i][j] = E.ddR[1][2][i][j];
  }
}

// x (t, Euler ZYX) from a float 4x4 (column-major) — estimateRigidTransformationNewton's initial state.
S3D_HD void state_from_matrix(const float T[16], double x[6]) {
  x[0] = T[12]; x[1] = T[13]; x[2] = T[14];
  x[3] = atan2((double)T[6], (double)T[10]);                 // atan2(T(2,1), T(2,2))
  x[4] = asin(fmin(1.0, fmax(-1.0, -(double)T[2])));         // asin(-T(2,0)), clamped
  x[5] = atan2((double)T[1], (double)T[0]);                  // atan2(T(1,0), T(0,0))
}

// applyState on the identity: T = [R(x) | t], rounded to float (column-major).
S3D_HD void matrix_from_state(const double x[6], float T[16]) {
  Euler E;
  euler_derivs(x, E, false);
  for (int c = 0; c < 3; ++c) { for (int r = 0; r < 3; ++r) T[c * 4 + r] = (float)E.R[r][c]; T[c * 4 + 3] = 0.f; }
  T[12] = (float)x[0]; T[13] = (float)x[1]; T[14] = (float)x[2]; T[15] = 1.f;
}

// f, gradient g[6] and exact Hessian H[6][6] of the GICP objective at x from the 74 sums of one evaluation pass
// (OptimizationFunctorWithIndices::operator() and ::dfddf).  Layout of `sums`:
//   [sym3(a,b)*10 + sym4(c,e)]  sum M[a][b] phi_c phi_e, phi = (p, 1)      x-independent for one correspondence set
//   [60 + a*4 + c]              sum (M d)[a] phi_c                            d = float(T(x) p) - q  exactly as PCL forms it
//   [72] sum d^T M d            [73] number of correspondences m
// One entry of the gradient (idx 0..5) or of the Hessian (idx 6 + 6 i + j), so that the GPU can spread the 42 entries over
// threads while the host (tests) walks them in a loop — the arithmetic per entry is the same.
S3D_HD double objective_entry(const double* sums, const Euler& E, int idx) {
  const double s = 2.0 / sums[73];
  if (idx < 3) return s * sums[60 + idx * 4 + 3];
  if (idx < 6) {
    const int k = idx - 3;
    double gr = 0;
    for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) gr += E.dR[k][a][b] * (s * sums[60 + a * 4 + b]);
    return gr;
  }
  int i = (idx - 6) / 6, j = (idx - 6) % 6;
  if (i < 3 && j < 3) return s * sums[sym3(i, j) * 10 + 9];
  if (i >= 3 && j < 3) { const int t = i; i = j; j = t; }
  if (i < 3) {  // translation-rotation block
    const int a = i, k = j - 3;
    double h = 0;
    for (int c = 0; c < 3; ++c) for (int b = 0; b < 3; ++b) h += E.dR[k][c][b] * (s * sums[sym3(a, c) * 10 + sym4(b, 3)]);
    return h;
  }
  const int k = i - 3, l = j - 3;  // rotation-rotation block: first-order part + second-derivative part
  double h = 0;
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) {
      for (int c = 0; c < 3; ++c) for (int e = 0; e < 3; ++e) h += E.dR[k][a][b] * E.dR[l][c][e] * (s * sums[sym3(a, c) * 10 + sym4(b, e)]);
      h += E.ddR[k][l][a][b] * (s * sums[60 + a * 4 + b]);
    }
  return h;
}

S3D_HD void objective_from_sums(const double* sums, const double x[6], double& f, double (&g)[6], double (&H)[6][6]) {
  Euler E;
  euler_derivs(x, E, true);
  f = sums[72] / sums[73];
  for (int i = 0; i < 6; ++i) g[i] = objective_entry(sums, E, i);
  for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) H[i][j] = objective_entry(sums, E, 6 + 6 * i + j);
}

// delta = H'^-1 g, H' = H with negative eigenvalues replaced by the largest one (PCL 1.14 Newton step).
// Positive-definite H (the normal case) is detected and solved by Cholesky, which is the same delta.
S3D_HD void newton_direction(const double (&H)[6][6], const double (&g)[6], double (&delta)[6]) {
  double L[6][6];
  bool pd = true;
  for (int i = 0; i < 6 && pd; ++i)
    for (int j = 0; j <= i; ++j) {
      double s = H[i][j];
      for (int k = 0; k < j; ++k) s -= L[i][k] * L[j][k];
      if (i == j) { if (!(s > 0.0)) { pd = false; break; } L[i][i] = sqrt(s); }
      else L[i][j] = s / L[j][j];
    }
  if (pd) {
    double y[6];
    for (int i = 0; i < 6; ++i) { double s = g[i]; for (int k = 0; k < i; ++k) s -= L[i][k] * y[k]; y[i] = s / L[i][i]; }
    for (int i = 5; i >= 0; --i) { double s = y[i]; for (int k = i + 1; k < 6; ++k) s -= L[k][i] * delta[k]; delta[i] = s / L[i][i]; }
    return;
  }
  double A[6][6], V[6][6], w[6];
  for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) A[i][j] = H[i][j];
  jacobi_eigen<6>(A, V, w);
  double wmax = w[0];
  for (int i = 1; i < 6; ++i) wmax = fmax(wmax, w[i]);
  for (int r = 0; r < 6; ++r) delta[r] = 0.0;
  for (int i = 0; i < 6; ++i) {
    const double inv = (w[i] < 0) ? 1.0 / wmax : 1.0 / w[i];
    double proj = 0;
    for (int r = 0; r < 6; ++r) proj += V[r][i] * g[r];
    for (int r = 0; r < 6; ++r) delta[r] += V[r][i] * (inv * proj);
  }
}

// estimateRigidTransformationNewton as a resumable state machine: every objective evaluation PCL's loop asks for is one
// data pass on the GPU (gicp.cu), so the optimiser yields whenever it needs f (and the sums for g, H) at a new state.
struct NewtonState {
  double x[6];        // accepted state
  double xc[6];       // state whose evaluation is pending / was just delivered
  double fcur, alpha;
  double g[6], H[6][6], delta[6];
  int it, ls, phase;  // phase: 0 = waiting for the evaluation at the start state, 1 = line search, 2 = finished
};

S3D_HD void newton_begin(NewtonState& st, const float T[16]) {
  state_from_matrix(T, st.x);
  for (int i = 0; i < 6; ++i) st.xc[i] = st.x[i];
  st.it = 0; st.ls = 0; st.alpha = 1.0; st.phase = 0;
}

S3D_HD bool newton_new_step(NewtonState& st) {  // do { ++it; direction; alpha = 1 ... }
  ++st.it;
  newton_direction(st.H, st.g, st.delta);
  st.alpha = 1.0; st.ls = 0;
  for (int r = 0; r < 6; ++r) st.xc[r] = st.x[r] - st.alpha * st.delta[r];
  st.phase = 1;
  return true;
}

// f, g, H = objective at st.xc (the evaluation that was pending).  Returns true when another evaluation (at the new st.xc)
// is needed, false when the optimiser is finished (result in st.x).  Mirrors PCL 1.14: back-tracking alpha = 1, 1/2, ...
// (10 trials) until f decreases, stop on no improvement, on both gradient norms < 1e-2, or after max_inner iterations.
S3D_HD bool newton_advance_pre(NewtonState& st, double f, const double (&g)[6], const double (&H)[6][6], int max_inner) {
  if (st.phase == 0 || (st.phase == 1 && f < st.fcur)) {
    const bool first = st.phase == 0;
    for (int r = 0; r < 6; ++r) { st.x[r] = st.xc[r]; st.g[r] = g[r]; for (int c = 0; c < 6; ++c) st.H[r][c] = H[r][c]; }
    st.fcur = f;
    if (first) return newton_new_step(st);
    const double gtn = sqrt(st.g[0] * st.g[0] + st.g[1] * st.g[1] + st.g[2] * st.g[2]);
    const double grn = sqrt(st.g[3] * st.g[3] + st.g[4] * st.g[4] + st.g[5] * st.g[5]);
    if (gtn < 1e-2 && grn < 1e-2) { st.phase = 2; return false; }  // translation_/rotation_gradient_tolerance_
    if (st.it < max_inner) return newton_new_step(st);
    st.phase = 2;
    return false;
  }
  if (st.phase == 1) {
    ++st.ls;
    st.alpha /= 2;
    if (st.ls < 10) {
      for (int r = 0; r < 6; ++r) st.xc[r] = st.x[r] - st.alpha * st.delta[r];
      return true;
    }
    st.phase = 2;  // no improvement found
    return false;
  }
  return false;
}

// ---- speculative back-tracking -------------------------------------------------------------------------------------
// PCL tries alpha = 1, 1/2, ..., 2^-9 one objective evaluation at a time.  On the GPU an evaluation is a data pass and
// a host poll, and the tail of the trials only runs in the float-rounding dominated regime near convergence, so trial 0
// is evaluated alone and, if it fails, trials 1..9 together in ONE pass; the first improving trial is then selected,
// which is exactly what the sequential loop would have accepted.
constexpr int kLineSearchTrials = 10;

S3D_HD void newton_trial_state(const NewtonState& st, int j, double xc[6]) {
  double alpha = 1.0;
  for (int i = 0; i < j; ++i) alpha /= 2;  // same halving sequence as the sequential loop (exact in binary)
  for (int r = 0; r < 6; ++r) xc[r] = st.x[r] - alpha * st.delta[r];
}

// f_trial[j] = f at trial j for j in [first, first + count).  Returns the accepted trial or -1.
S3D_HD int newton_pick_trial(const NewtonState& st, const double* f_trial, int first, int count) {
  for (int j = first; j < first + count; ++j) if (f_trial[j] < st.fcur) return j;
  return -1;
}

// Makes trial j the pending state, as if the sequential loop had just evaluated it.
S3D_HD void newton_select_trial(NewtonState& st, int j) {
  st.alpha = 1.0;
  for (int i = 0; i < j; ++i) st.alpha /= 2;
  st.ls = j;
  for (int r = 0; r < 6; ++r) st.xc[r] = st.x[r] - st.alpha * st.delta[r];
}

// `sums` = evaluation at st.xc (host-side convenience: computes the objective, then advances)
S3D_HD bool newton_advance(NewtonState& st, const double* sums, int max_inner) {
  double f, g[6], H[6][6];
  objective_from_sums(sums, st.xc, f, g, H);
  return newton_advance_pre(st, f, g, H, max_inner);
}

// Mahalanobis matrix of one correspondence (SURVEY A.4): M = (R C1 R^T + C2)^-1 with C = I - (1-eps) n n^T.
// RRt = R R^T (R comes from float matrices, so it is not exactly orthonormal), a = R n1, b = n2.  M: 6 unique (sym3 order).
S3D_HD void mahalanobis6(const double (&RRt)[3][3], const double a[3], const double b[3], double (&M)[6]) {
  const double k = 1.0 - kGicpEpsilon;
  double t[3][3];
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) t[i][j] = RRt[i][j] - k * a[i] * a[j] + ((i == j ? 1.0 : 0.0) - k * b[i] * b[j]);
  const double c00 = t[1][1] * t[2][2] - t[1][2] * t[2][1];
  const double c01 = t[0][2] * t[2][1] - t[0][1] * t[2][2];
  const double c02 = t[0][1] * t[1][2] - t[0][2] * t[1][1];
  const double c11 = t[0][0] * t[2][2] - t[0][2] * t[2][0];
  const double c12 = t[0][2] * t[1][0] - t[0][0] * t[1][2];
  const double c22 = t[0][0] * t[1][1] - t[0][1] * t[1][0];
  const double c10 = t[1][2] * t[2][0] - t[1][0] * t[2][2];
  const double c20 = t[1][0] * t[2][1] - t[1][1] * t[2][0];
  const double det = t[0][0] * c00 + t[0][1] * c10 + t[0][2] * c20;
  const double inv = 1.0 / det;
  M[0] = c00 * inv; M[1] = c01 * inv; M[2] = c02 * inv; M[3] = c11 * inv; M[4] = c12 * inv; M[5] = c22 * inv;
}

}  // namespace s3d

#include "gicp_bfgs.h"
