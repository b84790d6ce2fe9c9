// Host build of the DIRECT7 path of slam3d_b200/csrc/ndt_math.h for the CPU test-suite (tests/test_hostdirect7.py).
// Test-only: does on the host what ndt.cu does on the device for NDT_OMP with S3D_NDT_OMP_DIRECT7 (voxel keys, stable order
// inside a voxel, leaf finalisation and validity bit, the 7-cell lookup with float division, the 44 sums, the resumable
// optimiser), with plain sequential sums, so that it can be held bit for bit to the oracle without a GPU.
#include <algorithm>
#include <cmath>
#include <unordered_map>
#include <vector>

#include "../slam3d_b200/csrc/ndt_math.h"

namespace {
inline void transform_se3(const float* T, const float* p, float* o) {  // x*c0 + (y*c1 + (z*c2 + c3))
  o[0] = p[0] * T[0] + (p[1] * T[4] + (p[2] * T[8] + T[12]));
  o[1] = p[0] * T[1] + (p[1] * T[5] + (p[2] * T[9] + T[13]));
  o[2] = p[0] * T[2] + (p[1] * T[6] + (p[2] * T[10] + T[14]));
}
struct Grid {
  std::vector<s3d::NdtLeaf> leaves;              // leaves with >= 6 points (the device's hash holds exactly these)
  std::unordered_map<uint32_t, uint32_t> index;  // voxel key -> leaf
  float resolution, inv; int32_t min_b[3], div_b[3]; uint32_t mul1, mul2;
};
bool build_grid(const float* pts, int n, float resolution, Grid& G) {
  G.resolution = resolution;
  G.inv = 1.0f / resolution;
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int i = 0; i < n; ++i) for (int a = 0; a < 3; ++a) { mn[a] = std::min(mn[a], pts[4 * i + a]); mx[a] = std::max(mx[a], pts[4 * i + a]); }
  const long long dx = (long long)((mx[0] - mn[0]) * G.inv) + 1, dy = (long long)((mx[1] - mn[1]) * G.inv) + 1, dz = (long long)((mx[2] - mn[2]) * G.inv) + 1;
  if (dx * dy * dz > 2147483647ll) return false;
  for (int a = 0; a < 3; ++a) { G.min_b[a] = (int)std::floor(mn[a] * G.inv); G.div_b[a] = (int)std::floor(mx[a] * G.inv) - G.min_b[a] + 1; }
  G.mul1 = (uint32_t)G.div_b[0]; G.mul2 = (uint32_t)G.div_b[0] * (uint32_t)G.div_b[1];
  std::vector<std::pair<uint32_t, uint32_t>> kv(n);
  for (int i = 0; i < n; ++i) {
    const int i0 = (int)std::floor(pts[4 * i] * G.inv) - G.min_b[0], i1 = (int)std::floor(pts[4 * i + 1] * G.inv) - G.min_b[1], i2 = (int)std::floor(pts[4 * i + 2] * G.inv) - G.min_b[2];
    kv[i] = {(uint32_t)i0 + (uint32_t)i1 * G.mul1 + (uint32_t)i2 * G.mul2, (uint32_t)i};
  }
  std::stable_sort(kv.begin(), kv.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
  size_t i = 0;
  while (i < kv.size()) {
    size_t j = i + 1;
    while (j < kv.size() && kv[j].first == kv[i].first) ++j;
    const int nr = (int)(j - i);
    if (nr >= 6) {
      float cs[3] = {0, 0, 0}; double ms[3] = {0, 0, 0}, cov[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
      for (size_t l = i; l < j; ++l) {
        const float* p = pts + 4 * kv[l].second;
        const double d[3] = {p[0], p[1], p[2]};
        for (int a = 0; a < 3; ++a) { ms[a] += d[a]; cs[a] += p[a]; for (int b = 0; b < 3; ++b) cov[a][b] += d[a] * d[b]; }
      }
      s3d::NdtLeaf L;
      L.cx = cs[0] / (float)nr; L.cy = cs[1] / (float)nr; L.cz = cs[2] / (float)nr;
      const bool valid = s3d::ndt_finalize_leaf(nr, ms, cov, L.mean, L.icov) && s3d::ndt_icov_usable(L.icov);
      L.key = valid ? kv[i].first : (kv[i].first | s3d::kNdtLeafInvalid);
      G.index[kv[i].first] = (uint32_t)G.leaves.size();
      G.leaves.push_back(L);
    }
    i = j;
  }
  return true;
}
// the kept leaves of query q in offset order (what ndt_eval_kernel<true> collects)
int direct7(const Grid& G, const float q[3], uint32_t out[7], uint32_t keys[7]) {
  long long ijk[3];
  if (!s3d::ndt_direct7_cell(q[0], q[1], q[2], G.resolution, ijk)) return 0;
  int nc = 0;
  for (int i = 0; i < 7; ++i) {
    uint32_t key;
    if (!s3d::ndt_direct7_key(ijk, i, G.min_b, G.div_b, G.mul1, G.mul2, key)) continue;
    const auto it = G.index.find(key);
    if (it == G.index.end() || (G.leaves[it->second].key & s3d::kNdtLeafInvalid)) continue;
    keys[nc] = key;
    out[nc++] = it->second;
  }
  return nc;
}
void evaluate(const Grid& G, const float* src, int n, const float* T, const double x_eval[6], double d1, double d2, double* sums) {
  for (int i = 0; i < s3d::kNdtSums; ++i) sums[i] = 0.0;
  s3d::NdtAngular A;
  s3d::ndt_angle_derivatives(x_eval, A);
  for (int i = 0; i < n; ++i) {
    float q[3];
    transform_se3(T, src + 4 * i, q);
    uint32_t leaf[7], keys[7];
    const int nc = direct7(G, q, leaf, keys);
    if (!nc) continue;
    const double xo[3] = {src[4 * i], src[4 * i + 1], src[4 * i + 2]};
    s3d::NdtPointDerivs P;
    s3d::ndt_point_derivatives(A, xo, P);
    for (int k = 0; k < nc; ++k) {
      const s3d::NdtLeaf& L = G.leaves[leaf[k]];
      const double xt[3] = {(double)q[0] - L.mean[0], (double)q[1] - L.mean[1], (double)q[2] - L.mean[2]};
      s3d::ndt_accumulate(P, d1, d2, xt, L.icov, sums);
      sums[43] += 1.0;
    }
  }
}
}  // namespace

extern "C" {
// DIRECT7 keys of each query over the grid of `tgt` (n_tgt x 4 floats): keys[7 i + j], 0xFFFFFFFF past counts[i].
int hd_direct7_keys(const float* tgt, int n_tgt, float resolution, const float* q, int n_q, uint32_t* keys, int* counts) {
  Grid G;
  if (!build_grid(tgt, n_tgt, resolution, G)) return -1;
  for (int i = 0; i < n_q; ++i) {
    uint32_t leaf[7], k[7];
    counts[i] = direct7(G, q + 4 * i, leaf, k);
    for (int j = 0; j < 7; ++j) keys[7 * i + j] = j < counts[i] ? k[j] : 0xFFFFFFFFu;
  }
  return (int)G.leaves.size();
}
// pcl_source (moving, n_src x 4 floats), pcl_target (voxelised, n_tgt x 4 floats), guess column-major float 4x4.
// out: T[16] final_transformation_, info = {converged, nr_iterations, line_iterations, n_pairs_last, evaluations, n_leaves}
int hd_ndt_register(const float* src, int n_src, const float* tgt, int n_tgt, const float* guess, float resolution, double step_size,
                    double outlier_ratio, double trans_eps, int max_iter, float* T_out, int* info) {
  Grid G;
  for (int i = 0; i < 16; ++i) T_out[i] = (i % 5 == 0) ? 1.f : 0.f;
  for (int i = 0; i < 6; ++i) info[i] = 0;
  if (!build_grid(tgt, n_tgt, resolution, G) || G.leaves.empty()) return 0;
  info[5] = (int)G.leaves.size();
  double d1, d2;
  s3d::ndt_gauss_constants((double)resolution, outlier_ratio, d1, d2);
  float T[16];
  for (int i = 0; i < 16; ++i) T[i] = guess[i];
  double x0[6];
  s3d::ndt_initial_state(T, x0);
  s3d::NdtOptState st;
  s3d::ndt_opt_begin(st, x0, step_size, trans_eps, max_iter);
  double sums[s3d::kNdtSums];
  int evals = 0;
  for (;;) {
    evaluate(G, src, n_src, T, st.x_t, d1, d2, sums);
    ++evals;
    if (!s3d::ndt_opt_on_eval(st, sums)) break;
    s3d::ndt_convert_transform(st.x_t, T);
  }
  for (int i = 0; i < 16; ++i) T_out[i] = T[i];
  info[0] = st.converged; info[1] = st.nr_iterations; info[2] = st.line_iterations; info[3] = (int)st.n_pairs_last; info[4] = evals;
  return 0;
}
}
