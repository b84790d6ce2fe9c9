// ndt_math.h — scalar FP64 math of the NDT branch, callable from host and device.
//
// What it computes (reference: pcl::NormalDistributionsTransform as driven by slam3d doNDT,
// slam3d/sensor/pcl/PointCloudSensor.cpp:84-117; [Magnusson 2009] eq. 6.9-6.21, [More, Thuente 1994]):
//   * a voxel's Gaussian from its point sums (VoxelGridCovariance::applyFilter second pass: single-pass covariance,
//     eigenvalue inflation to 1 % of the largest, inverse);
//   * the angular / per-point derivative tables and one (point, voxel) contribution to score, gradient and Hessian
//     (computeAngleDerivatives, computePointDerivatives, updateDerivatives);
//   * the outer Newton loop of computeTransformation with the More-Thuente line search of computeStepLengthMT as a
//     RESUMABLE state machine: ndt_opt_on_eval() consumes the 44 sums of one pass over the moving cloud and either asks
//     for the next evaluation (a float 4x4) or finishes.  On the GPU one thread per registration runs it between two
//     evaluation kernels; the CPU test-suite (tests/hostmath.cpp) runs the very same code against the oracle.
// B200-first design note: PCL evaluates the line search's later trials without the Hessian and recomputes it afterwards
// (computeHessian) with the same per-term arithmetic; here every pass produces score, gradient and Hessian, so the
// recomputation pass disappears and the values are the same.
#pragma once

#include "gicp_math.h"

#if defined(__CUDACC__)
#define S3D_UNROLL _Pragma("unroll")
#else
#define S3D_UNROLL
#endif

namespace s3d {

constexpr int kNdtSums = 44;  // [0] score, [1..6] gradient, [7 + 6 i + j] Hessian, [43] number of (point, voxel) pairs

// One voxel of the target grid (VoxelGridCovariance::Leaf).  cx,cy,cz = float centroid (a point of voxel_centroids_),
// key = PCL's linear voxel index (ascending order == order of the centroid cloud), nr < 6: not part of the centroid cloud.
// A leaf of >= 6 points that applyFilter marked invalid (nr_points = -1) carries kNdtLeafInvalid in its key: the radius search
// still returns it, DIRECT7 does not.  PCL forms the index as an int, so bit 31 is free on every grid where PCL's arithmetic is
// defined.
struct NdtLeaf {
  float cx, cy, cz;
  uint32_t key;
  double mean[3];
  double icov[9];  // row-major (not exactly symmetric, as in PCL)
};

constexpr uint32_t kNdtLeafInvalid = 0x80000000u;

S3D_HD void ndt_inv3(const double (&a)[3][3], double (&c)[3][3]) {  // Eigen 3x3 inverse: cofactors / determinant
  c[0][0] = a[1][1] * a[2][2] - a[1][2] * a[2][1];
  c[0][1] = a[0][2] * a[2][1] - a[0][1] * a[2][2];
  c[0][2] = a[0][1] * a[1][2] - a[0][2] * a[1][1];
  c[1][0] = a[1][2] * a[2][0] - a[1][0] * a[2][2];
  c[1][1] = a[0][0] * a[2][2] - a[0][2] * a[2][0];
  c[1][2] = a[0][2] * a[1][0] - a[0][0] * a[1][2];
  c[2][0] = a[1][0] * a[2][1] - a[1][1] * a[2][0];
  c[2][1] = a[0][1] * a[2][0] - a[0][0] * a[2][1];
  c[2][2] = a[0][0] * a[1][1] - a[0][1] * a[1][0];
  const double det = a[0][0] * c[0][0] + a[0][1] * c[1][0] + a[0][2] * c[2][0];
  const double inv = 1.0 / det;
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) c[i][j] *= inv;
}

// Second pass of VoxelGridCovariance::applyFilter for one leaf with nr >= min_points_per_voxel_ (6).
// ms = sum of the points, cs = sum of the outer products (both double, input order).  Returns false when PCL marks
// the leaf invalid (icov stays the constructor's zero matrix; the leaf still takes part in the radius search).
S3D_HD bool ndt_finalize_leaf(int nr, const double ms[3], const double (&cs)[3][3], double mean[3], double icov[9]) {
  const double dn = (double)nr;
  for (int a = 0; a < 3; ++a) mean[a] = ms[a] / dn;
  const double f = (dn - 1.0) / dn;
  double cov[3][3];
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) cov[a][b] = ((cs[a][b] - 2.0 * (ms[a] * mean[b])) / dn + mean[a] * mean[b]) * f;
  double A[3][3], V[3][3], w[3];
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) A[i][j] = i >= j ? cov[i][j] : cov[j][i];  // SelfAdjointEigenSolver reads the lower triangle
  jacobi_eigen<3>(A, V, w);
  int o[3] = {0, 1, 2};  // ascending eigenvalues (bubble sort, same as the oracle)
  for (int a = 0; a < 2; ++a) for (int b = 0; b < 2 - a; ++b) if (w[o[b]] > w[o[b + 1]]) { const int t = o[b]; o[b] = o[b + 1]; o[b + 1] = t; }
  double ev[3] = {w[o[0]], w[o[1]], w[o[2]]};
  for (int i = 0; i < 9; ++i) icov[i] = 0.0;
  if (ev[0] < -1e-12 || ev[1] < -1e-12 || ev[2] <= 0) return false;
  const double min_ev = 0.01 * ev[2];  // min_covar_eigvalue_mult_
  if (ev[0] < min_ev) {
    ev[0] = min_ev;
    if (ev[1] < min_ev) ev[1] = min_ev;
    double E[3][3], VD[3][3], Vi[3][3], D[3][3];
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) { E[r][c] = V[r][o[c]]; D[r][c] = r == c ? ev[r] : 0.0; }
    mat3_mul(E, D, VD);
    ndt_inv3(E, Vi);
    mat3_mul(VD, Vi, cov);  // evecs * eigen_val * evecs.inverse()
  }
  double ic[3][3];
  ndt_inv3(cov, ic);
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) icov[3 * r + c] = ic[r][c];
  return true;
}

// nr_points >= 0 after applyFilter for a leaf ndt_finalize_leaf accepted: PCL also marks the leaf invalid when
// icov_.maxCoeff() == inf or icov_.minCoeff() == -inf (folded as std::max / std::min over the row-major entries, as the oracle does)
S3D_HD bool ndt_icov_usable(const double icov[9]) {
  double mx = -1.7976931348623157e308, mn = 1.7976931348623157e308;
  for (int i = 0; i < 9; ++i) { mx = mx < icov[i] ? icov[i] : mx; mn = icov[i] < mn ? icov[i] : mn; }
  return !(mx == INFINITY || mn == -INFINITY);
}

// ---- pclomp DIRECT7 neighbourhood (VoxelGridCovariance::getNeighborhoodAtPoint7) -------------------------------------------
// Offsets in pclomp's order; a query reads its own voxel and the 6 face neighbours, each once, in this order.
S3D_HD int ndt_direct7_offset(int i, int axis) {
  return i == 0 ? 0 : ((i - 1) / 2 == axis ? ((i & 1) ? 1 : -1) : 0);
}

// ijk = (int) floor(p / leaf_size) per axis, float DIVISION (not applyFilter's * inverse_leaf_size).  Returns false for a
// non-finite coordinate or a cell index outside int32 (PCL's cast is undefined there; here such a point has no neighbours).
S3D_HD bool ndt_direct7_cell(float x, float y, float z, float leaf, long long ijk[3]) {
  const float p[3] = {x, y, z};
  for (int a = 0; a < 3; ++a) {
#if defined(__CUDA_ARCH__)
    const float f = floorf(__fdiv_rn(p[a], leaf));
#else
    const float f = floorf(p[a] / leaf);
#endif
    if (!(f >= -2147483648.0f && f < 2147483648.0f)) return false;
    ijk[a] = (long long)f;
  }
  return true;
}

// The linear index (ijk + d - min_b) . divb_mul of offset i, or false when min_b <= ijk + d <= max_b fails on some axis
// (max_b = min_b + div_b - 1).  The caller keeps the leaf under that key only if it exists with nr_points >= 6 and valid.
S3D_HD bool ndt_direct7_key(const long long ijk[3], int i, const int32_t min_b[3], const int32_t div_b[3], uint32_t mul1, uint32_t mul2,
                            uint32_t& key) {
  long long c[3];
  for (int a = 0; a < 3; ++a) {
    c[a] = ijk[a] + ndt_direct7_offset(i, a) - min_b[a];
    if (c[a] < 0 || c[a] >= div_b[a]) return false;
  }
  key = (uint32_t)c[0] + (uint32_t)c[1] * mul1 + (uint32_t)c[2] * mul2;
  return true;
}

struct NdtAngular { double aj[8][3]; double ah[15][3]; };  // angular_jacobian_ / angular_hessian_ (the 4th column multiplies 0)

S3D_HD void ndt_angle_derivatives(const double x[6], NdtAngular& A) {
  double cx, cy, cz, sx, sy, sz;
  if (fabs(x[3]) < 10e-5) { cx = 1.0; sx = 0.0; } else { cx = cos(x[3]); sx = sin(x[3]); }
  if (fabs(x[4]) < 10e-5) { cy = 1.0; sy = 0.0; } else { cy = cos(x[4]); sy = sin(x[4]); }
  if (fabs(x[5]) < 10e-5) { cz = 1.0; sz = 0.0; } else { cz = cos(x[5]); sz = sin(x[5]); }
  A.aj[0][0] = (-sx * sz + cx * sy * cz); A.aj[0][1] = (-sx * cz - cx * sy * sz); A.aj[0][2] = (-cx * cy);
  A.aj[1][0] = (cx * sz + sx * sy * cz);  A.aj[1][1] = (cx * cz - sx * sy * sz);  A.aj[1][2] = (-sx * cy);
  A.aj[2][0] = (-sy * cz);                A.aj[2][1] = sy * sz;                   A.aj[2][2] = cy;
  A.aj[3][0] = sx * cy * cz;              A.aj[3][1] = (-sx * cy * sz);           A.aj[3][2] = sx * sy;
  A.aj[4][0] = (-cx * cy * cz);           A.aj[4][1] = cx * cy * sz;              A.aj[4][2] = (-cx * sy);
  A.aj[5][0] = (-cy * sz);                A.aj[5][1] = (-cy * cz);                A.aj[5][2] = 0;
  A.aj[6][0] = (cx * cz - sx * sy * sz);  A.aj[6][1] = (-cx * sz - sx * sy * cz); A.aj[6][2] = 0;
  A.aj[7][0] = (sx * cz + cx * sy * sz);  A.aj[7][1] = (cx * sy * cz - sx * sz);  A.aj[7][2] = 0;
  A.ah[0][0] = (-cx * sz - sx * sy * cz);  A.ah[0][1] = (-cx * cz + sx * sy * sz);  A.ah[0][2] = sx * cy;
  A.ah[1][0] = (-sx * sz + cx * sy * cz);  A.ah[1][1] = (-cx * sy * sz - sx * cz);  A.ah[1][2] = (-cx * cy);
  A.ah[2][0] = (cx * cy * cz);             A.ah[2][1] = (-cx * cy * sz);            A.ah[2][2] = (cx * sy);
  A.ah[3][0] = (sx * cy * cz);             A.ah[3][1] = (-sx * cy * sz);            A.ah[3][2] = (sx * sy);
  A.ah[4][0] = (-sx * cz - cx * sy * sz);  A.ah[4][1] = (sx * sz - cx * sy * cz);   A.ah[4][2] = 0;
  A.ah[5][0] = (cx * cz - sx * sy * sz);   A.ah[5][1] = (-sx * sy * cz - cx * sz);  A.ah[5][2] = 0;
  A.ah[6][0] = (-cy * cz);                 A.ah[6][1] = (cy * sz);                  A.ah[6][2] = (-sy);
  A.ah[7][0] = (-sx * sy * cz);            A.ah[7][1] = (sx * sy * sz);             A.ah[7][2] = (sx * cy);
  A.ah[8][0] = (cx * sy * cz);             A.ah[8][1] = (-cx * sy * sz);            A.ah[8][2] = (-cx * cy);
  A.ah[9][0] = (sy * sz);                  A.ah[9][1] = (sy * cz);                  A.ah[9][2] = 0;
  A.ah[10][0] = (-sx * cy * sz);           A.ah[10][1] = (-sx * cy * cz);           A.ah[10][2] = 0;
  A.ah[11][0] = (cx * cy * sz);            A.ah[11][1] = (cx * cy * cz);            A.ah[11][2] = 0;
  A.ah[12][0] = (-cy * cz);                A.ah[12][1] = (cy * sz);                 A.ah[12][2] = 0;
  A.ah[13][0] = (-cx * sz - sx * sy * cz); A.ah[13][1] = (-cx * cz + sx * sy * sz); A.ah[13][2] = 0;
  A.ah[14][0] = (-sx * sz + cx * sy * cz); A.ah[14][1] = (-cx * sy * sz - sx * cz); A.ah[14][2] = 0;
}

// computePointDerivatives: the 8 non-trivial Jacobian entries and the 15 Hessian entries of one (untransformed) point
struct NdtPointDerivs { double j[8]; double h[15]; };

S3D_HD void ndt_point_derivatives(const NdtAngular& A, const double x[3], NdtPointDerivs& P) {
  for (int r = 0; r < 8; ++r) P.j[r] = (A.aj[r][0] * x[0] + A.aj[r][1] * x[1]) + A.aj[r][2] * x[2];
  for (int r = 0; r < 15; ++r) P.h[r] = (A.ah[r][0] * x[0] + A.ah[r][1] * x[1]) + A.ah[r][2] * x[2];
}

S3D_HD double ndt_dot3(const double a[3], const double b[3]) { return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]; }
S3D_HD void ndt_mv3(const double* ci, const double v[3], double o[3]) {  // ci row-major 3x3
  for (int r = 0; r < 3; ++r) o[r] = (ci[3 * r] * v[0] + ci[3 * r + 1] * v[1]) + ci[3 * r + 2] * v[2];
}

// updateDerivatives for one (point, voxel) pair: acc[0] += score_inc, acc[1..6] += gradient, acc[7..42] += Hessian.
// xt = transformed point - voxel mean, ci = the voxel's inverse covariance.
S3D_HD void ndt_accumulate(const NdtPointDerivs& P, double gauss_d1, double gauss_d2, const double xt[3], const double* ci, double* acc) {
  double cx[3];
  ndt_mv3(ci, xt, cx);
  double e = exp(-gauss_d2 * ndt_dot3(xt, cx) / 2);
  const double score_inc = -gauss_d1 * e;
  e = gauss_d2 * e;
  if (e > 1 || e < 0 || e != e) return;  // "Error checking for invalid values": contributes nothing, not even the score
  e *= gauss_d1;
  acc[0] += score_inc;
  // point_jacobian_ columns: e0 e1 e2 | (0, j0, j1) | (j2, j3, j4) | (j5, j6, j7)
  double col[6][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}, {0, P.j[0], P.j[1]}, {P.j[2], P.j[3], P.j[4]}, {P.j[5], P.j[6], P.j[7]}};
  double cj[6][3], xcj[6];
  S3D_UNROLL
  for (int i = 0; i < 6; ++i) { ndt_mv3(ci, col[i], cj[i]); xcj[i] = ndt_dot3(xt, cj[i]); }
  // x^T Sigma^-1 (second derivative vector) for the 6 distinct vectors a b c d e f of eq. 6.21
  double hv[6][3] = {{0, P.h[0], P.h[1]}, {0, P.h[2], P.h[3]}, {0, P.h[4], P.h[5]}, {P.h[6], P.h[7], P.h[8]}, {P.h[9], P.h[10], P.h[11]}, {P.h[12], P.h[13], P.h[14]}};
  double xch[6];
  S3D_UNROLL
  for (int k = 0; k < 6; ++k) { double t[3]; ndt_mv3(ci, hv[k], t); xch[k] = ndt_dot3(xt, t); }
  S3D_UNROLL
  for (int i = 0; i < 6; ++i) {
    acc[1 + i] += xcj[i] * e;
    S3D_UNROLL
    for (int j = 0; j < 6; ++j) {
      double second = 0.0;  // x^T Sigma^-1 point_hessian_.block<3,1>(3 i, j): a b c / b d e / c e f for i, j >= 3
      if (i >= 3 && j >= 3) {
        const int a = i - 3, b = j - 3;
        const int k = a == 0 ? b : (b == 0 ? a : (a == 1 && b == 1 ? 3 : (a == 2 && b == 2 ? 5 : 4)));
        second = xch[k];
      }
      acc[7 + 6 * i + j] += e * ((-gauss_d2 * xcj[i] * xcj[j] + second) + ndt_dot3(col[j], cj[i]));
    }
  }
}

// float(cos(double(a))): the correctly rounded float cosine (definition shared with the oracle)
S3D_HD float ndt_cosf(float a) { return (float)cos((double)a); }
S3D_HD float ndt_sinf(float a) { return (float)sin((double)a); }

// convertTransform(x, Matrix4f): Translation3f * AngleAxisf(x3, X) * AngleAxisf(x4, Y) * AngleAxisf(x5, Z), float products
// left to right, ((a0 b0 + a1 b1) + a2 b2).  T column-major.
S3D_HD void ndt_convert_transform(const double x[6], float T[16]) {
  float R[3][3][3];
  for (int axis = 0; axis < 3; ++axis) {
    const float ang = (float)x[3 + axis];
    const float s = ndt_sinf(ang), c = ndt_cosf(ang);
    const int i = (axis + 1) % 3, j = (axis + 2) % 3;
    for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) R[axis][a][b] = 0.f;
#if defined(__CUDA_ARCH__)
    R[axis][axis][axis] = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, c), 1.0f), c);
    R[axis][i][j] = __fsub_rn(0.f, s);
    R[axis][j][i] = __fadd_rn(0.f, s);
#else
    R[axis][axis][axis] = (1.0f - c) * 1.0f + c;
    R[axis][i][j] = 0.f - s;
    R[axis][j][i] = 0.f + s;
#endif
    R[axis][i][i] = c; R[axis][j][j] = c;
  }
  float A[3][3], B[3][3];
#if defined(__CUDA_ARCH__)
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c)
    A[r][c] = __fadd_rn(__fadd_rn(__fmul_rn(R[0][r][0], R[1][0][c]), __fmul_rn(R[0][r][1], R[1][1][c])), __fmul_rn(R[0][r][2], R[1][2][c]));
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c)
    B[r][c] = __fadd_rn(__fadd_rn(__fmul_rn(A[r][0], R[2][0][c]), __fmul_rn(A[r][1], R[2][1][c])), __fmul_rn(A[r][2], R[2][2][c]));
#else
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) A[r][c] = (R[0][r][0] * R[1][0][c] + R[0][r][1] * R[1][1][c]) + R[0][r][2] * R[1][2][c];
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) B[r][c] = (A[r][0] * R[2][0][c] + A[r][1] * R[2][1][c]) + A[r][2] * R[2][2][c];
#endif
  for (int c = 0; c < 3; ++c) { for (int r = 0; r < 3; ++r) T[c * 4 + r] = B[r][c]; T[c * 4 + 3] = 0.f; }
  T[12] = (float)x[0]; T[13] = (float)x[1]; T[14] = (float)x[2]; T[15] = 1.f;
}

// JacobiSVD<Matrix6d>(H).solve(b): one-sided Jacobi SVD, pseudo-inverse with Eigen's default threshold (6 eps sigma_max)
S3D_HD void ndt_svd_solve6(const double (&Hin)[6][6], const double b[6], double x[6]) {
  double A[6][6], V[6][6];
  for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) { A[i][j] = Hin[i][j]; V[i][j] = i == j ? 1.0 : 0.0; }
  for (int sweep = 0; sweep < 60; ++sweep) {
    bool rotated = false;
    for (int p = 0; p < 5; ++p)
      for (int q = p + 1; q < 6; ++q) {
        double alpha = 0, beta = 0, gamma = 0;
        for (int k = 0; k < 6; ++k) { alpha += A[k][p] * A[k][p]; beta += A[k][q] * A[k][q]; gamma += A[k][p] * A[k][q]; }
        if (gamma == 0.0 || fabs(gamma) <= 1e-15 * sqrt(alpha * beta)) continue;
        rotated = true;
        const double zeta = (beta - alpha) / (2.0 * gamma);
        const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
        for (int k = 0; k < 6; ++k) {
          const double ap = A[k][p], aq = A[k][q];
          A[k][p] = c * ap - s * aq; A[k][q] = s * ap + c * aq;
          const double vp = V[k][p], vq = V[k][q];
          V[k][p] = c * vp - s * vq; V[k][q] = s * vp + c * vq;
        }
      }
    if (!rotated) break;
  }
  double sv[6], smax = 0;
  for (int j = 0; j < 6; ++j) { double s = 0; for (int k = 0; k < 6; ++k) s += A[k][j] * A[k][j]; sv[j] = sqrt(s); if (sv[j] > smax) smax = sv[j]; }
  const double thr = smax * 6.0 * 2.220446049250313e-16;
  for (int i = 0; i < 6; ++i) x[i] = 0;
  for (int j = 0; j < 6; ++j) {
    if (!(sv[j] > thr) || sv[j] == 0.0) continue;
    double ub = 0;
    for (int k = 0; k < 6; ++k) ub += A[k][j] * b[k];
    const double coef = ub / (sv[j] * sv[j]);
    for (int i = 0; i < 6; ++i) x[i] += V[i][j] * coef;
  }
}

S3D_HD bool ndt_update_interval(double& a_l, double& f_l, double& g_l, double& a_u, double& f_u, double& g_u, double a_t, double f_t, double g_t) {
  if (f_t > f_l) { a_u = a_t; f_u = f_t; g_u = g_t; return false; }
  if (g_t * (a_l - a_t) > 0) { a_l = a_t; f_l = f_t; g_l = g_t; return false; }
  if (g_t * (a_l - a_t) < 0) { a_u = a_l; f_u = f_l; g_u = g_l; a_l = a_t; f_l = f_t; g_l = g_t; return false; }
  return true;
}

S3D_HD double ndt_trial_value(double a_l, double f_l, double g_l, double a_u, double f_u, double g_u, double a_t, double f_t, double g_t) {
  if (a_t == a_l && a_t == a_u) return a_t;
  int cond;
  if (a_t == a_l) cond = 4;
  else if (f_t > f_l) cond = 1;
  else if (g_t * g_l < 0) cond = 2;
  else if (fabs(g_t) <= fabs(g_l)) cond = 3;
  else cond = 4;
  if (cond == 4) {
    const double z = 3 * (f_t - f_u) / (a_t - a_u) - g_t - g_u;
    const double w = sqrt(z * z - g_t * g_u);
    return a_u + (a_t - a_u) * (w - g_u - z) / (g_t - g_u + 2 * w);
  }
  const double z = 3 * (f_t - f_l) / (a_t - a_l) - g_t - g_l;
  const double w = sqrt(z * z - g_t * g_l);
  const double a_c = a_l + (a_t - a_l) * (w - g_l - z) / (g_t - g_l + 2 * w);
  if (cond == 1) {
    const double a_q = a_l - 0.5 * (a_l - a_t) * g_l / (g_l - (f_l - f_t) / (a_l - a_t));
    if (fabs(a_c - a_l) < fabs(a_q - a_l)) return a_c;
    return 0.5 * (a_q + a_c);
  }
  const double a_s = a_l - (a_l - a_t) / (g_l - g_t) * g_l;
  if (cond == 2) return fabs(a_c - a_t) >= fabs(a_s - a_t) ? a_c : a_s;
  const double a_t_next = fabs(a_c - a_t) < fabs(a_s - a_t) ? a_c : a_s;
  if (a_t > a_l) return fmin(a_t + 0.66 * (a_u - a_t), a_t_next);
  return fmax(a_t + 0.66 * (a_u - a_t), a_t_next);
}

// State of computeTransformation + computeStepLengthMT between two evaluations.
struct NdtOptState {
  double x[6];               // `transform`
  double x_t[6];             // state of the pending / last evaluation
  double score, g[6], H[6][6];
  double step_dir[6];
  double phi_0, d_phi_0, a_l, f_l, g_l, a_u, f_u, g_u, a_t;
  double step_max, step_min, trans_eps;
  int32_t interval_converged, open_interval, step_iterations;
  int32_t phase;             // 0: first computeDerivatives pending, 1: first trial of a line search pending, 2: later trial pending, 3: finished
  int32_t nr_iterations, max_iterations, converged, line_iterations;
  uint32_t n_pairs_last, reserved;
};

S3D_HD void ndt_opt_begin(NdtOptState& st, const double x0[6], double step_size, double trans_eps, int max_iterations) {
  for (int i = 0; i < 6; ++i) { st.x[i] = x0[i]; st.x_t[i] = x0[i]; st.step_dir[i] = 0; st.g[i] = 0; for (int j = 0; j < 6; ++j) st.H[i][j] = 0; }
  st.score = 0;
  st.phi_0 = st.d_phi_0 = st.a_l = st.f_l = st.g_l = st.a_u = st.f_u = st.g_u = st.a_t = 0;
  st.step_max = step_size; st.step_min = trans_eps / 2; st.trans_eps = trans_eps;
  st.interval_converged = 0; st.open_interval = 1; st.step_iterations = 0;
  st.phase = 0; st.nr_iterations = 0; st.max_iterations = max_iterations; st.converged = 0; st.line_iterations = 0;
  st.n_pairs_last = 0; st.reserved = 0;
}

// Tail of one outer iteration (after the line search returned a_t) and head of the next one, repeated while no evaluation
// is needed.  Returns true when an evaluation at st.x_t is pending.
S3D_HD bool ndt_opt_next_outer(NdtOptState& st, double a_t, bool first) {
  for (;;) {
    if (!first) {
      double delta[6];
      for (int i = 0; i < 6; ++i) delta[i] = st.step_dir[i] * a_t;   // delta *= delta_norm
      float Tinc[16];
      ndt_convert_transform(delta, Tinc);                              // transformation_
      for (int i = 0; i < 6; ++i) st.x[i] += delta[i];                // transform += delta
      const float t0 = Tinc[12], t1 = Tinc[13], t2 = Tinc[14];
#if defined(__CUDA_ARCH__)
      const double translation_sqr = (double)__fadd_rn(__fmul_rn(t0, t0), __fadd_rn(__fmul_rn(t1, t1), __fmul_rn(t2, t2)));
#else
      const double translation_sqr = (double)(t0 * t0 + (t1 * t1 + t2 * t2));
#endif
      st.nr_iterations += 1;
      // transformation_rotation_epsilon_ is 0 (never set by slam3d): only the translation clause can fire
      if (st.nr_iterations >= st.max_iterations || (st.trans_eps > 0 && translation_sqr <= st.trans_eps)) { st.converged = 1; st.phase = 3; return false; }
    }
    first = false;
    double neg_g[6], delta[6];
    for (int i = 0; i < 6; ++i) neg_g[i] = -st.g[i];
    ndt_svd_solve6(st.H, neg_g, delta);
    double nn = 0;
    for (int i = 0; i < 6; ++i) nn += delta[i] * delta[i];
    const double delta_norm = sqrt(nn);
    if (delta_norm == 0 || delta_norm != delta_norm) { st.converged = delta_norm != delta_norm ? 1 : 0; st.phase = 3; return false; }
    for (int i = 0; i < 6; ++i) st.step_dir[i] = delta[i] / delta_norm;
    // computeStepLengthMT prologue
    st.phi_0 = -st.score;
    double d = 0;
    for (int i = 0; i < 6; ++i) d += st.g[i] * st.step_dir[i];
    st.d_phi_0 = -d;
    if (st.d_phi_0 >= 0) {
      if (st.d_phi_0 == 0) { a_t = 0; continue; }  // "return 0": the iteration ends with a zero step
      st.d_phi_0 *= -1;
      for (int i = 0; i < 6; ++i) st.step_dir[i] *= -1;
    }
    const double mu = 1.e-4;
    st.step_iterations = 0;
    st.a_l = 0; st.a_u = 0;
    st.f_l = st.phi_0 - st.phi_0 - mu * st.d_phi_0 * st.a_l; st.g_l = st.d_phi_0 - mu * st.d_phi_0;
    st.f_u = st.phi_0 - st.phi_0 - mu * st.d_phi_0 * st.a_u; st.g_u = st.d_phi_0 - mu * st.d_phi_0;
    st.interval_converged = (st.step_max - st.step_min) < 0 ? 1 : 0;
    st.open_interval = 1;
    double at = delta_norm;
    at = fmin(at, st.step_max);
    at = fmax(at, st.step_min);
    st.a_t = at;
    for (int i = 0; i < 6; ++i) st.x_t[i] = st.x[i] + st.step_dir[i] * at;
    st.phase = 1;
    return true;
  }
}

// Consumes the sums of the evaluation at st.x_t.  Returns true when another evaluation (at the new st.x_t) is needed.
S3D_HD bool ndt_opt_on_eval(NdtOptState& st, const double* sums) {
  st.score = sums[0];
  for (int i = 0; i < 6; ++i) { st.g[i] = sums[1 + i]; for (int j = 0; j < 6; ++j) st.H[i][j] = sums[7 + 6 * i + j]; }
  st.n_pairs_last = sums[43] < 4294967295.0 ? (uint32_t)sums[43] : 0xFFFFFFFFu;
  if (st.phase == 0) return ndt_opt_next_outer(st, 0.0, true);
  const double mu = 1.e-4, nu = 0.9;
  const double phi_t = -st.score;
  double d = 0;
  for (int i = 0; i < 6; ++i) d += st.g[i] * st.step_dir[i];
  const double d_phi_t = -d;
  const double psi_t = phi_t - st.phi_0 - mu * st.d_phi_0 * st.a_t;
  const double d_psi_t = d_phi_t - mu * st.d_phi_0;
  if (st.phase == 2) {  // tail of the loop body of computeStepLengthMT
    if (st.open_interval && (psi_t <= 0 && d_psi_t >= 0)) {
      st.open_interval = 0;
      st.f_l += st.phi_0 - mu * st.d_phi_0 * st.a_l; st.g_l += mu * st.d_phi_0;
      st.f_u += st.phi_0 - mu * st.d_phi_0 * st.a_u; st.g_u += mu * st.d_phi_0;
    }
    if (st.open_interval) st.interval_converged = ndt_update_interval(st.a_l, st.f_l, st.g_l, st.a_u, st.f_u, st.g_u, st.a_t, psi_t, d_psi_t) ? 1 : 0;
    else st.interval_converged = ndt_update_interval(st.a_l, st.f_l, st.g_l, st.a_u, st.f_u, st.g_u, st.a_t, phi_t, d_phi_t) ? 1 : 0;
    st.step_iterations += 1;
  }
  if (!st.interval_converged && st.step_iterations < 10 && !(psi_t <= 0 && d_phi_t <= -nu * st.d_phi_0)) {
    double at;
    if (st.open_interval) at = ndt_trial_value(st.a_l, st.f_l, st.g_l, st.a_u, st.f_u, st.g_u, st.a_t, psi_t, d_psi_t);
    else at = ndt_trial_value(st.a_l, st.f_l, st.g_l, st.a_u, st.f_u, st.g_u, st.a_t, phi_t, d_phi_t);
    at = fmin(at, st.step_max);
    at = fmax(at, st.step_min);
    st.a_t = at;
    for (int i = 0; i < 6; ++i) st.x_t[i] = st.x[i] + st.step_dir[i] * at;
    st.phase = 2;
    return true;
  }
  st.line_iterations += st.step_iterations;
  return ndt_opt_next_outer(st, st.a_t, false);
}

// Host only: the initial `transform` vector of computeTransformation from final_transformation_ (= guess, float):
// translation and Matrix3f::eulerAngles(0, 1, 2) (Eigen 3.3/3.4, first angle in [0, pi]) with the host libm's float
// functions — evaluated on the host so that the CUDA path and the oracle see the same bits.
inline void ndt_initial_state(const float T[16], double x[6]) {
  const float kPi = 3.14159265358979323846f;
  const float m00 = T[0], m01 = T[4], m02 = T[8], m10 = T[1], m11 = T[5], m12 = T[9], m20 = T[2], m21 = T[6], m22 = T[10];
  float r0 = atan2f(m12, m22);
  const float c2 = sqrtf(m00 * m00 + m01 * m01);
  float r1;
  if (r0 > 0.f) { r0 -= kPi; r1 = atan2f(-m02, -c2); }
  else r1 = atan2f(-m02, c2);
  const float s1 = sinf(r0), c1 = cosf(r0);
  const float r2 = atan2f(s1 * m20 - c1 * m10, c1 * m11 - s1 * m21);
  x[0] = (double)T[12]; x[1] = (double)T[13]; x[2] = (double)T[14];
  x[3] = (double)(-r0); x[4] = (double)(-r1); x[5] = (double)(-r2);
}

// gauss_d1_, gauss_d2_ (eq. 6.8), host libm
inline void ndt_gauss_constants(double resolution, double outlier_ratio, double& d1, double& d2) {
  const double c1 = 10.0 * (1 - outlier_ratio);
  const double c2 = outlier_ratio / pow(resolution, 3);
  const double d3 = -log(c2);
  d1 = -log(c1 + c2) - d3;
  d2 = -2 * log((-log(c1 * exp(-0.5) + c2) - d3) / d1);
}

}  // namespace s3d
