// ndt_omp_oracle.cpp — CPU ORACLE of registration_algorithm = NDT_OMP with pclomp's default DIRECT7 neighbour search, a library
// of its own beside libs3d_oracle.so (loaded by oracle/ndt_omp.py; TEST INFRASTRUCTURE, PARITY UNPINNED — see the header of
// s3d_oracle.cpp).  It compiles s3d_oracle.cpp into itself and reuses its NDT restatement (ndt_oracle.inc: VoxelGridCovariance,
// derivatives, More-Thuente, convertTransform, fitness); only the neighbour search of computeDerivatives / computeHessian, and
// the drivers that call it, are restated here.  Built like s3d_oracle.cpp: g++ -O2 -std=c++17 -ffp-contract=off -fno-fast-math.
//
// Restates, from upstream source (koide3/ndt_omp; slam3d/sensor/pcl/PointCloudSensor.cpp:84-117 doNDT, :153-157 case NDT_OMP):
//   pclomp::NormalDistributionsTransform with search_method = DIRECT7, its default (doNDT never calls
//   setNeighborhoodSearchMethod): computeDerivatives and computeHessian call VoxelGridCovariance::getNeighborhoodAtPoint7(x_trans_pt)
//   = PCL's getNeighborhoodAtPoint(relative_coordinates, point, neighbors) with 7 offsets, instead of kdtree_.radiusSearch.
//
// Choices upstream leaves open, fixed here (the CUDA path, slam3d_b200/csrc/ndt_math.h, makes the same ones):
//   * offset order (0,0,0), (+1,0,0), (-1,0,0), (0,+1,0), (0,-1,0), (0,0,+1), (0,0,-1): the column order of pclomp's
//     relative_coordinates; the leaves' contributions are added in this order;
//   * ijk = (int) floor(p / leaf_size_) with a float DIVISION, as getNeighborhoodAtPoint writes it, while applyFilter keys the
//     voxels with p * inverse_leaf_size_: at a cell face the two may disagree, and the division is what is restated;
//   * a query with a non-finite coordinate or a cell index outside int32 has no neighbours (PCL's cast is undefined there);
//   * an offset is kept when min_b_ <= ijk + d <= max_b_ on every axis and its leaf exists in leaves_ with nr_points >= 6
//     (min_points_per_voxel_): this drops sparse voxels and the leaves applyFilter marked invalid (nr_points = -1), which the
//     radius search does return;
//   * sums run point by point, each point's neighbours in offset order.  pclomp sums per OpenMP thread and then adds the thread
//     sums, so a real pclomp run is reproducible only to rounding, and only up to that rounding is this its restatement.
// Unpinned, and outside this restatement: pclomp forks the NDT of PCL 1.8, while ndt_oracle.inc restates PCL 1.14's.  Anything
// that changed between the two in ndt.hpp / voxel_grid_covariance.hpp (the exits of computeTransformation, the convergence flag
// of a zero or NaN step, the eigenvalue inflation of applyFilter, float versus double in the transform conversions) may differ
// in pclomp and is taken from PCL 1.14 here.

#include "s3d_oracle.cpp"

namespace {

// The parts of VoxelGridCovariance that getNeighborhoodAtPoint reads besides leaves_: leaf_size_, min_b_, max_b_, divb_mul_
// (applyFilter's prologue, as in ndt_build_grid).
struct Direct7Grid {
  const NdtGrid* grid = nullptr;
  float leaf_size = 0.f;
  int64_t min_b[3] = {0, 0, 0}, max_b[3] = {0, 0, 0}, divb_mul[3] = {0, 0, 0};
};

static void direct7_grid(const std::vector<P4>& cloud, float resolution, const NdtGrid& G, Direct7Grid& D) {
  D.grid = &G;
  D.leaf_size = resolution;
  if (G.centroids.empty()) return;
  const float inv = 1.0f / resolution;
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  for (const P4& p : cloud) {
    if (!finite3(p)) continue;
    mn[0] = std::min(mn[0], p.x); mx[0] = std::max(mx[0], p.x);
    mn[1] = std::min(mn[1], p.y); mx[1] = std::max(mx[1], p.y);
    mn[2] = std::min(mn[2], p.z); mx[2] = std::max(mx[2], p.z);
  }
  for (int a = 0; a < 3; ++a) {
    D.min_b[a] = static_cast<int>(std::floor(mn[a] * inv));
    D.max_b[a] = static_cast<int>(std::floor(mx[a] * inv));
  }
  D.divb_mul[0] = 1;
  D.divb_mul[1] = D.max_b[0] - D.min_b[0] + 1;
  D.divb_mul[2] = D.divb_mul[1] * (D.max_b[1] - D.min_b[1] + 1);
}

// getNeighborhoodAtPoint7(point): the kept leaves (as Cand ids into G.leaves, d2 unused) in offset order
static void direct7_search(const Direct7Grid& D, const P4& q, std::vector<KdTree::Cand>& out) {
  out.clear();
  static const int kOff[7][3] = {{0, 0, 0}, {1, 0, 0}, {-1, 0, 0}, {0, 1, 0}, {0, -1, 0}, {0, 0, 1}, {0, 0, -1}};
  const std::vector<NdtLeaf>& leaves = D.grid->leaves;
  const float pq[3] = {q.x, q.y, q.z};
  int64_t ijk[3];
  for (int a = 0; a < 3; ++a) {
    const float f = std::floor(pq[a] / D.leaf_size);
    if (!(f >= -2147483648.0f && f < 2147483648.0f)) return;
    ijk[a] = static_cast<int64_t>(f);
  }
  for (int i = 0; i < 7; ++i) {
    bool inside = true;
    int64_t idx = 0;
    for (int a = 0; a < 3; ++a) {
      const int64_t c = ijk[a] + kOff[i][a];
      if (c < D.min_b[a] || c > D.max_b[a]) inside = false;
      idx += (c - D.min_b[a]) * D.divb_mul[a];
    }
    if (!inside) continue;
    // leaves_.find(idx): leaves with < 6 points are not kept in G.leaves, and would fail the nr_points test below anyway
    const auto it = std::lower_bound(leaves.begin(), leaves.end(), static_cast<uint32_t>(idx),
                                     [](const NdtLeaf& L, uint32_t k) { return L.leaf_idx < k; });
    if (it == leaves.end() || it->leaf_idx != static_cast<uint32_t>(idx) || it->nr_points < 6) continue;
    out.push_back({0.f, static_cast<uint32_t>(it - leaves.begin())});
  }
}

// ndt_compute_derivatives / ndt_compute_hessian of ndt_oracle.inc with the DIRECT7 neighbourhood
static double direct7_compute_derivatives(NdtProblem& P, const Direct7Grid& D, double g[6], double H[6][6], const std::vector<P4>& trans_cloud,
                                          const double x[6], bool compute_hessian) {
  for (int i = 0; i < 6; ++i) { g[i] = 0; for (int j = 0; j < 6; ++j) H[i][j] = 0; }
  double score = 0;
  ndt_angle_derivatives(P.S, x);
  std::vector<KdTree::Cand> nb;
  P.n_pairs_last = 0;
  for (size_t idx = 0; idx < P.input->size(); ++idx) {
    const P4& xt_pt = trans_cloud[idx];
    direct7_search(D, xt_pt, nb);
    const P4& xp = (*P.input)[idx];
    const double xo[3] = {xp.x, xp.y, xp.z};
    for (const KdTree::Cand& c : nb) {
      const NdtLeaf& L = P.grid->leaves[c.id];
      const double xt[3] = {static_cast<double>(xt_pt.x) - L.mean[0], static_cast<double>(xt_pt.y) - L.mean[1], static_cast<double>(xt_pt.z) - L.mean[2]};
      ndt_point_derivatives(P.S, xo);
      score += ndt_update(P.S, g, H, xt, L.icov, true, compute_hessian);
      ++P.n_pairs_last;
    }
  }
  return score;
}

static void direct7_compute_hessian(NdtProblem& P, const Direct7Grid& D, double H[6][6], const std::vector<P4>& trans_cloud) {
  for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) H[i][j] = 0;
  std::vector<KdTree::Cand> nb;
  double g_unused[6];
  for (size_t idx = 0; idx < P.input->size(); ++idx) {
    const P4& xt_pt = trans_cloud[idx];
    direct7_search(D, xt_pt, nb);
    const P4& xp = (*P.input)[idx];
    const double xo[3] = {xp.x, xp.y, xp.z};
    for (const KdTree::Cand& c : nb) {
      const NdtLeaf& L = P.grid->leaves[c.id];
      const double xt[3] = {static_cast<double>(xt_pt.x) - L.mean[0], static_cast<double>(xt_pt.y) - L.mean[1], static_cast<double>(xt_pt.z) - L.mean[2]};
      ndt_point_derivatives(P.S, xo);
      ndt_update(P.S, g_unused, H, xt, L.icov, false, true);
    }
  }
}

// ndt_step_length of ndt_oracle.inc (computeStepLengthMT) on the DIRECT7 derivatives
static double direct7_step_length(NdtProblem& P, const Direct7Grid& D, const double x[6], double step_dir[6], double step_init, double step_max,
                                  double step_min, double& score, double g[6], double H[6][6], std::vector<P4>& trans_cloud, M4f& final_T,
                                  int& line_iterations) {
  const double phi_0 = -score;
  double d_phi_0 = 0;
  for (int i = 0; i < 6; ++i) d_phi_0 += g[i] * step_dir[i];
  d_phi_0 = -d_phi_0;
  if (d_phi_0 >= 0) {
    if (d_phi_0 == 0) return 0;
    d_phi_0 *= -1;
    for (int i = 0; i < 6; ++i) step_dir[i] *= -1;
  }
  const int max_step_iterations = 10;
  int step_iterations = 0;
  const double mu = 1.e-4, nu = 0.9;
  double a_l = 0, a_u = 0;
  double f_l = ndt_psi(a_l, phi_0, phi_0, d_phi_0, mu), g_l = ndt_dpsi(d_phi_0, d_phi_0, mu);
  double f_u = ndt_psi(a_u, phi_0, phi_0, d_phi_0, mu), g_u = ndt_dpsi(d_phi_0, d_phi_0, mu);
  bool interval_converged = (step_max - step_min) < 0, open_interval = true;
  double a_t = step_init;
  a_t = std::min(a_t, step_max);
  a_t = std::max(a_t, step_min);
  double x_t[6];
  auto evaluate = [&](bool compute_hessian) {
    for (int i = 0; i < 6; ++i) x_t[i] = x[i] + step_dir[i] * a_t;
    final_T = ndt_convert_transform(x_t);
    for (size_t i = 0; i < P.input->size(); ++i) trans_cloud[i] = transform_se3(final_T, (*P.input)[i]);
    score = direct7_compute_derivatives(P, D, g, H, trans_cloud, x_t, compute_hessian);
  };
  evaluate(true);
  double phi_t = -score, d_phi_t = 0;
  for (int i = 0; i < 6; ++i) d_phi_t += g[i] * step_dir[i];
  d_phi_t = -d_phi_t;
  double psi_t = ndt_psi(a_t, phi_t, phi_0, d_phi_0, mu), d_psi_t = ndt_dpsi(d_phi_t, d_phi_0, mu);
  while (!interval_converged && step_iterations < max_step_iterations && !(psi_t <= 0 && d_phi_t <= -nu * d_phi_0)) {
    if (open_interval) a_t = ndt_trial_value(a_l, f_l, g_l, a_u, f_u, g_u, a_t, psi_t, d_psi_t);
    else a_t = ndt_trial_value(a_l, f_l, g_l, a_u, f_u, g_u, a_t, phi_t, d_phi_t);
    a_t = std::min(a_t, step_max);
    a_t = std::max(a_t, step_min);
    evaluate(false);
    phi_t = -score;
    d_phi_t = 0;
    for (int i = 0; i < 6; ++i) d_phi_t += g[i] * step_dir[i];
    d_phi_t = -d_phi_t;
    psi_t = ndt_psi(a_t, phi_t, phi_0, d_phi_0, mu);
    d_psi_t = ndt_dpsi(d_phi_t, d_phi_0, mu);
    if (open_interval && (psi_t <= 0 && d_psi_t >= 0)) {
      open_interval = false;
      f_l += phi_0 - mu * d_phi_0 * a_l; g_l += mu * d_phi_0;
      f_u += phi_0 - mu * d_phi_0 * a_u; g_u += mu * d_phi_0;
    }
    if (open_interval) interval_converged = ndt_update_interval(a_l, f_l, g_l, a_u, f_u, g_u, a_t, psi_t, d_psi_t);
    else interval_converged = ndt_update_interval(a_l, f_l, g_l, a_u, f_u, g_u, a_t, phi_t, d_phi_t);
    ++step_iterations;
  }
  if (step_iterations) direct7_compute_hessian(P, D, H, trans_cloud);
  line_iterations += step_iterations;
  return a_t;
}

// ndt_register of ndt_oracle.inc (align + computeTransformation + getFitnessScore) on the DIRECT7 derivatives
static void direct7_register(const std::vector<P4>& pcl_source, const std::vector<P4>& pcl_target, const M4f& guess,
                             const s3d_registration_parameters& cfg, NdtOutput& out) {
  const size_t N = pcl_source.size();
  NdtGrid G;
  ndt_build_grid(pcl_target, cfg.resolution, G);
  Direct7Grid D;
  direct7_grid(pcl_target, cfg.resolution, G, D);
  KdTree tree_target;
  tree_target.build(pcl_target.data(), pcl_target.size());
  out.converged = false; out.outer_iterations = 0; out.inner_iterations = 0; out.n_corr = 0;
  M4f final_T = m4f_identity();
  if (!G.centroids.empty()) {  // "Voxel grid is not searchable" otherwise
    NdtProblem P;
    P.input = &pcl_source; P.grid = &G;
    std::memset(&P.S, 0, sizeof P.S);
    const double res = static_cast<double>(cfg.resolution);
    const double c1 = 10.0 * (1 - cfg.outlier_ratio);
    const double c2 = cfg.outlier_ratio / std::pow(res, 3);
    const double d3 = -std::log(c2);
    P.S.gauss_d1 = -std::log(c1 + c2) - d3;
    P.S.gauss_d2 = -2 * std::log((-std::log(c1 * std::exp(-0.5) + c2) - d3) / P.S.gauss_d1);
    P.S.r2 = static_cast<float>(res * res);
    for (int r = 0; r < 3; ++r) P.S.pj[r][r] = 1.0;
    std::vector<P4> trans_cloud(pcl_source);
    for (size_t i = 0; i < N; ++i) trans_cloud[i].w = 1.0f;
    bool guess_is_identity = true;
    for (int i = 0; i < 16; ++i) if (guess.m[i] != ((i % 5 == 0) ? 1.f : 0.f)) guess_is_identity = false;
    if (!guess_is_identity) {
      final_T = guess;
      for (size_t i = 0; i < N; ++i) trans_cloud[i] = transform_se3(guess, trans_cloud[i]);
    }
    double x[6], g[6], H[6][6];
    float eul[3];
    ndt_euler_angles_012(final_T, eul);
    for (int r = 0; r < 3; ++r) { x[r] = static_cast<double>(final_T(r, 3)); x[3 + r] = static_cast<double>(eul[r]); }
    double score = direct7_compute_derivatives(P, D, g, H, trans_cloud, x, true);
    while (!out.converged) {
      double neg_g[6], delta[6];
      for (int i = 0; i < 6; ++i) neg_g[i] = -g[i];
      ndt_svd_solve6(H, neg_g, delta);
      double nn = 0;
      for (int i = 0; i < 6; ++i) nn += delta[i] * delta[i];
      double delta_norm = std::sqrt(nn);
      if (delta_norm == 0 || std::isnan(delta_norm)) { out.converged = std::isnan(delta_norm); break; }
      for (int i = 0; i < 6; ++i) delta[i] /= delta_norm;
      delta_norm = direct7_step_length(P, D, x, delta, delta_norm, cfg.step_size, cfg.transformation_epsilon / 2, score, g, H, trans_cloud,
                                       final_T, out.inner_iterations);
      for (int i = 0; i < 6; ++i) delta[i] *= delta_norm;
      const M4f Tinc = ndt_convert_transform(delta);
      for (int i = 0; i < 6; ++i) x[i] += delta[i];
      const float t0 = Tinc(0, 3), t1 = Tinc(1, 3), t2 = Tinc(2, 3);
      const double translation_sqr = static_cast<double>(t0 * t0 + (t1 * t1 + t2 * t2));
      ++out.outer_iterations;
      if (out.outer_iterations >= cfg.maximum_iterations || (cfg.transformation_epsilon > 0 && translation_sqr <= cfg.transformation_epsilon))
        out.converged = true;
    }
    out.n_corr = static_cast<uint32_t>(std::min<uint64_t>(P.n_pairs_last, 0xFFFFFFFFu));
  }
  out.final_T = final_T;
  double sum = 0; int nr = 0;
  for (size_t i = 0; i < N; ++i) {
    const P4 q = transform_se3(out.final_T, pcl_source[i]);
    KdTree::Cand nn;
    tree_target.knn(q, 1, &nn);
    if (static_cast<double>(nn.d2) <= cfg.max_correspondence_distance) { sum += nn.d2; ++nr; }
  }
  out.fitness = nr > 0 ? sum / nr : std::numeric_limits<double>::max();
}

}  // namespace

extern "C" {

// align(source, target, guess, config) with registration_algorithm = NDT_OMP in a slam3d build with pclomp (DIRECT7): the
// voxel filter, the <100 gate, doNDT and the gates of align_impl in s3d_oracle.cpp.  guess column-major.
int s3d_oracle_ndt_omp_align(s3d_cloud source, s3d_cloud target, const double guess[16], const s3d_registration_parameters* cfg,
                             s3d_result* res) {
  std::memset(res, 0, sizeof *res);
  for (int i = 0; i < 16; ++i) res->T[i] = (i % 5 == 0) ? 1.0 : 0.0;
  const P4* src = reinterpret_cast<const P4*>(source.xyzw);
  const P4* tgt = reinterpret_cast<const P4*>(target.xyzw);
  std::vector<P4> fsrc, ftgt;
  if (cfg->point_cloud_density > 0) {
    voxel_filter(src, source.n, static_cast<float>(cfg->point_cloud_density), fsrc, nullptr, nullptr);
    voxel_filter(tgt, target.n, static_cast<float>(cfg->point_cloud_density), ftgt, nullptr, nullptr);
  } else {
    fsrc.assign(src, src + source.n);
    ftgt.assign(tgt, tgt + target.n);
  }
  res->n_source = static_cast<uint32_t>(fsrc.size());
  res->n_target = static_cast<uint32_t>(ftgt.size());
  if (ftgt.size() < 100 || fsrc.size() < 100) {
    g_err = "Too few points after filtering, you may have to decrease 'point_cloud_density'.";
    return res->status = S3D_TOO_FEW_POINTS;
  }
  M4f guess_f;
  for (int i = 0; i < 16; ++i) guess_f.m[i] = static_cast<float>(guess[i]);
  NdtOutput out{};
  direct7_register(ftgt, fsrc, guess_f, *cfg, out);  // ndt.setInputSource(target); ndt.setInputTarget(source)
  for (int i = 0; i < 16; ++i) res->T[i] = static_cast<double>(out.final_T.m[i]);
  res->fitness = out.fitness;
  res->converged = out.converged ? 1 : 0;
  res->outer_iterations = out.outer_iterations;
  res->inner_iterations = out.inner_iterations;
  res->n_correspondences = out.n_corr;
  if (!out.converged || out.fitness > cfg->max_fitness_score) {
    g_err = "NDT failed with Fitness-Score " + std::to_string(out.fitness) + " > " + std::to_string(cfg->max_fitness_score);
    return res->status = S3D_NOT_CONVERGED;
  }
  double ginv[16], delta[16];
  iso_inverse(guess, ginv);
  m4d_mul(ginv, res->T, delta);
  const double tn = std::sqrt(delta[12] * delta[12] + delta[13] * delta[13] + delta[14] * delta[14]);
  if (tn > cfg->max_translation || rotation_angle(delta) > cfg->max_rotation) {
    g_err = "ICP result is to far away from guess";
    return res->status = S3D_TOO_FAR_FROM_GUESS;
  }
  return res->status = S3D_OK;
}

// Test hook: the DIRECT7 neighbourhood of each query over the VoxelGridCovariance of `target` at `resolution`: keys[7 i + j] =
// PCL's linear index of the j-th kept leaf in offset order (0xFFFFFFFF past counts[i]).  Returns the number of centroids.
int s3d_oracle_ndt_direct7_keys(s3d_cloud target, float resolution, s3d_cloud queries, uint32_t* keys, int32_t* counts) {
  std::vector<P4> tgt(reinterpret_cast<const P4*>(target.xyzw), reinterpret_cast<const P4*>(target.xyzw) + target.n);
  NdtGrid G;
  ndt_build_grid(tgt, resolution, G);
  Direct7Grid D;
  direct7_grid(tgt, resolution, G, D);
  const P4* q = reinterpret_cast<const P4*>(queries.xyzw);
  std::vector<KdTree::Cand> nb;
  for (size_t i = 0; i < queries.n; ++i) {
    for (int j = 0; j < 7; ++j) keys[7 * i + j] = 0xFFFFFFFFu;
    counts[i] = 0;
    if (G.centroids.empty()) continue;
    direct7_search(D, q[i], nb);
    for (const KdTree::Cand& c : nb) keys[7 * i + counts[i]++] = G.leaves[c.id].leaf_idx;
  }
  return static_cast<int>(G.centroids.size());
}

}  // extern "C"
