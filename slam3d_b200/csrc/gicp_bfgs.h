// gicp_bfgs.h — the inner GICP optimiser of PCL <= 1.13 (estimateRigidTransformationBFGS on pcl/registration/bfgs.h, a port
// of GSL's vector_bfgs2 with Fletcher's line search) as a resumable state machine, callable from host and device.  Included by
// gicp_math.h; the GPU loop (gicp.cu) runs it when a context selects S3D_GICP_BFGS.
//
// A port of bfgs_oracle.inc (the CPU test oracle), operation for operation (same expressions, same operand order, same constants).  Where the
// oracle calls the objective, the machine yields instead: it names the state xc = x0 + alpha p it needs, and the caller delivers
// f and the gradient there, both from the 13 residual sums of ONE evaluation pass.  The oracle asks for the gradient only at an
// alpha whose f it has just evaluated, and the point a line search accepts is that last alpha, so every request is one pass and
// no point is evaluated twice (the oracle's re-evaluations at the accepted point recompute the same numbers; reusing the sums
// of the pass is exact, while a second pass could round differently).
//
// S3D_BFGS_HIT(k), empty by default, marks the decisions of the line search (BfgsBranch) so that a host test can check that its
// cases exercise all of them.
#pragma once

#ifndef S3D_BFGS_HIT
#define S3D_BFGS_HIT(k) ((void)0)
#endif

namespace s3d {

// decision points of the machine (S3D_BFGS_HIT)
enum BfgsBranch {
  kHitBracketRho = 0,       // bracketing ends on the rho (sufficient decrease) test or on f not decreasing
  kHitBracketSlope = 1,     // bracketing ends on fpalpha >= 0
  kHitBracketWolfe = 2,     // Wolfe success inside bracketing
  kHitSectionWolfe = 3,     // Wolfe success inside sectioning
  kHitRoundoff = 4,         // sectioning stops: roundoff prevents progress (kNoProgress)
  kHitCubic = 5,            // interpolate: cubic through two values and two slopes
  kHitQuadratic = 6,        // interpolate: quadratic (no slope at b)
  kHitMaxInner = 7,         // the solve stops at it == max_inner while still running (PCL accepts the state)
  kHitGradient = 8,         // testGradient: |g| < 1e-2
  kHitDegenerate = 9,       // minimizeOneStep refuses to start: pnorm, g0norm or fp0 is 0 (kNoProgress)
  kHitLineSearchCap = 10,   // bracket_iters / section_iters exhausted (step length left at 0)
  kBfgsBranches = 11
};

// bfgs.h / GSL vector_bfgs2 constants (BFGS::Parameters) and estimateRigidTransformationBFGS's gradient tolerance
constexpr double kBfgsSigma = 0.01, kBfgsRho = 0.01, kBfgsTau1 = 9, kBfgsTau2 = 0.05, kBfgsTau3 = 0.5, kBfgsStepSize = 1;
constexpr int kBfgsOrder = 3, kBfgsBracketIters = 100, kBfgsSectionIters = 100;
constexpr double kBfgsGradientTol = 1e-2;
constexpr double kDblEpsilon = 2.220446049250313080847263336181640625e-16;  // std::numeric_limits<double>::epsilon()

enum BfgsStatus { kBfgsRunning = -1, kBfgsSuccess = 0, kBfgsNoProgress = 1 };
enum BfgsStage { kBfgsStart = 0, kBfgsBracket = 1, kBfgsSection = 2, kBfgsDone = 3 };

struct BfgsState {
  double x[6];                          // accepted state; the result once stage == kBfgsDone
  double xc[6];                         // state whose evaluation is pending: x0 + alpha p (x itself for kBfgsStart)
  double x0[6], g0[6], p[6];            // start of the step, its gradient, unit search direction
  double f, g0norm, pnorm, fp0, delta_f;
  // locals of BFGS::lineSearch that live across evaluations (f0 of the line search is `f`, which it does not change)
  double alpha, alpha_prev, falpha_prev, fpalpha_prev;
  double a, b, fa, fb, fpa, fpb;        // fpb is NaN when the bracket has no slope at b
  int i;                                // line-search iterations, one counter for bracketing and sectioning as in bfgs.h
  int it;                               // BFGS iterations of this solve (inner iterations)
  int stage;                            // BfgsStage
  int failed;                           // estimateRigidTransformationBFGS would throw (SolverDidntConvergeException)
};

S3D_HD double bfgs_dot6(const double* a, const double* b) { double s = 0; for (int i = 0; i < 6; ++i) s += a[i] * b[i]; return s; }
S3D_HD double bfgs_norm6(const double* a) { return sqrt(bfgs_dot6(a, a)); }
S3D_HD double bfgs_cubic(double c0, double c1, double c2, double c3, double z) { return c0 + z * (c1 + z * (c2 + z * c3)); }

// BFGS::interpolate — minimum of the cubic (or, without a derivative at b, quadratic) through (a, fa, fpa), (b, fb[, fpb]) on [xmin, xmax]
S3D_HD double bfgs_interpolate(double a, double fa, double fpa, double b, double fb, double fpb, double xmin, double xmax, int order) {
  double ymin = (xmin - a) / (b - a), ymax = (xmax - a) / (b - a);
  if (ymin > ymax) { const double t = ymin; ymin = ymax; ymax = t; }
  double y, fm;
  if (order > 2 && fpb == fpb && isfinite(fpb)) {
    S3D_BFGS_HIT(kHitCubic);
    fpa *= (b - a); fpb *= (b - a);
    const double eta = 3 * (fb - fa) - 2 * fpa - fpb, xi = fpa + fpb - 2 * (fb - fa);
    const double c0 = fa, c1 = fpa, c2 = eta, c3 = xi;
    y = ymin; fm = bfgs_cubic(c0, c1, c2, c3, ymin);
    { const double v = bfgs_cubic(c0, c1, c2, c3, ymax); if (v < fm) { y = ymax; fm = v; } }
    // roots of the derivative c1 + 2 c2 z + 3 c3 z^2
    const double qa = 3 * c3, qb = 2 * c2, qc = c1;
    if (qa == 0) {
      if (qb != 0) {
        const double z0 = -qc / qb;
        if (z0 > ymin && z0 < ymax) { const double v = bfgs_cubic(c0, c1, c2, c3, z0); if (v < fm) { y = z0; fm = v; } }
      }
    } else {
      const double disc = qb * qb - 4 * qa * qc;
      if (disc > 0) {
        const double t = -0.5 * (qb + (qb > 0 ? 1.0 : -1.0) * sqrt(disc));  // stable form
        double z0 = t / qa, z1 = (t != 0) ? qc / t : z0;
        if (z0 > z1) { const double s = z0; z0 = z1; z1 = s; }
        if (z0 > ymin && z0 < ymax) { const double v = bfgs_cubic(c0, c1, c2, c3, z0); if (v < fm) { y = z0; fm = v; } }
        if (z1 > ymin && z1 < ymax) { const double v = bfgs_cubic(c0, c1, c2, c3, z1); if (v < fm) { y = z1; fm = v; } }
      } else if (disc == 0) {
        const double z0 = -0.5 * qb / qa;
        if (z0 > ymin && z0 < ymax) { const double v = bfgs_cubic(c0, c1, c2, c3, z0); if (v < fm) { y = z0; fm = v; } }
      }
    }
  } else {
    S3D_BFGS_HIT(kHitQuadratic);
    fpa *= (b - a);
    const double fl = fa + ymin * (fpa + ymin * (fb - fa - fpa));
    const double fh = fa + ymax * (fpa + ymax * (fb - fa - fpa));
    const double c = 2 * (fb - fa - fpa);  // curvature
    y = ymin; fm = fl;
    if (fh < fm) { y = ymax; fm = fh; }
    if (c > a) {  // sic: bfgs.h compares the curvature with `a` where GSL has 0
      const double z = -fpa / c;
      if (z > ymin && z < ymax) { const double v = fa + z * (fpa + z * (fb - fa - fpa)); if (v < fm) { y = z; fm = v; } }
    }
  }
  return a + y * (b - a);
}

S3D_HD void bfgs_begin(BfgsState& st, const float T[16]) {  // the state estimateRigidTransformationBFGS starts from
  state_from_matrix(T, st.x);
  for (int i = 0; i < 6; ++i) st.xc[i] = st.x[i];
  st.it = 0; st.i = 0; st.stage = kBfgsStart; st.failed = 0;
}

S3D_HD bool bfgs_finish(BfgsState& st, int result, int max_inner) {
  if (result == kBfgsRunning && st.it == max_inner) S3D_BFGS_HIT(kHitMaxInner);
  st.failed = (result == kBfgsNoProgress || result == kBfgsSuccess || st.it == max_inner) ? 0 : 1;
  st.stage = kBfgsDone;
  return false;
}

S3D_HD void bfgs_set_trial(BfgsState& st) {  // the pending trial state, formed as the oracle forms it
  for (int i = 0; i < 6; ++i) st.xc[i] = st.x0[i] + st.alpha * st.p[i];
}

// BFGS::minimizeOneStep after the line search accepted alpha (f_new, g_new: objective at x0 + alpha p), then testGradient and the
// iteration cap of estimateRigidTransformationBFGS's loop.  true: another step follows; false: the solve is over.
S3D_HD bool bfgs_accept(BfgsState& st, double alpha, double f_new, const double* g_new, int max_inner) {
  double g[6], x[6];
  for (int i = 0; i < 6; ++i) g[i] = g_new[i];
  const double f0 = st.f;
  for (int i = 0; i < 6; ++i) x[i] = st.x0[i] + alpha * st.p[i];  // updatePosition
  st.f = f_new;
  st.delta_f = st.f - f0;
  // BFGS update of the direction: p' = g1 - A dx - B dg,  B = dx.g / dx.dg,  A = -(1 + dg.dg / dx.dg) B + dg.g / dx.dg
  double dx0[6], dg0[6];
  for (int i = 0; i < 6; ++i) { dx0[i] = x[i] - st.x0[i]; dg0[i] = g[i] - st.g0[i]; }
  const double dxg = bfgs_dot6(dx0, g), dgg = bfgs_dot6(dg0, g), dxdg = bfgs_dot6(dx0, dg0), dgnorm = bfgs_norm6(dg0);
  double A = 0, B = 0;
  if (dxdg != 0) { B = dxg / dxdg; A = -(1.0 + dgnorm * dgnorm / dxdg) * B + dgg / dxdg; }
  for (int i = 0; i < 6; ++i) st.p[i] = -A * dx0[i] + g[i] - B * dg0[i];
  for (int i = 0; i < 6; ++i) { st.g0[i] = g[i]; st.x0[i] = x[i]; st.x[i] = x[i]; }
  st.g0norm = bfgs_norm6(st.g0);
  st.pnorm = bfgs_norm6(st.p);
  const double pg = bfgs_dot6(st.p, g);
  const double dir = (pg >= 0.0) ? -1.0 : +1.0;
  for (int i = 0; i < 6; ++i) st.p[i] *= dir / st.pnorm;
  st.pnorm = bfgs_norm6(st.p);
  st.fp0 = bfgs_dot6(st.p, st.g0);
  if (bfgs_norm6(g) < kBfgsGradientTol) { S3D_BFGS_HIT(kHitGradient); return bfgs_finish(st, kBfgsSuccess, max_inner); }
  if (st.it < max_inner) return true;
  return bfgs_finish(st, kBfgsRunning, max_inner);
}

// Runs the optimiser from `go` to its next objective evaluation (true, at st.xc) or to the end of the solve (false).
enum BfgsGo { kGoStep = 0, kGoBracket = 1, kGoSection = 2 };
S3D_HD bool bfgs_run(BfgsState& st, int go, int max_inner) {
  for (;;) {
    if (go == kGoStep) {  // ++it; BFGS::minimizeOneStep up to the line search
      ++st.it;
      if (st.pnorm == 0.0 || st.g0norm == 0.0 || st.fp0 == 0.0) { S3D_BFGS_HIT(kHitDegenerate); return bfgs_finish(st, kBfgsNoProgress, max_inner); }
      double alpha1;
      if (st.delta_f < 0) {
        const double u = -st.delta_f, v = 10 * kDblEpsilon * fabs(st.f);
        const double del = (u < v) ? v : u;                   // std::max(u, v)
        const double w = 2.0 * del / (-st.fp0);
        alpha1 = (w < 1.0) ? w : 1.0;                         // std::min(1.0, w)
      } else {
        alpha1 = fabs(kBfgsStepSize);
      }
      st.alpha = alpha1; st.alpha_prev = 0.0;
      st.a = 0.0; st.b = st.alpha; st.fa = st.f; st.fb = 0.0; st.fpa = st.fp0; st.fpb = 0.0;
      st.falpha_prev = st.f; st.fpalpha_prev = st.fp0;
      st.i = 0;
      go = kGoBracket;
    }
    if (go == kGoBracket) {  // bracketing: f (and the slope) at alpha
      if (st.i++ < kBfgsBracketIters) { bfgs_set_trial(st); st.stage = kBfgsBracket; return true; }
      go = kGoSection;
    }
    // sectioning of [a, b]
    if (st.i++ < kBfgsSectionIters) {
      const double delta = st.b - st.a;
      st.alpha = bfgs_interpolate(st.a, st.fa, st.fpa, st.b, st.fb, st.fpb, st.a + kBfgsTau2 * delta, st.b - kBfgsTau3 * delta, kBfgsOrder);
      // the oracle evaluates f(alpha) before this test, which does not read it: that evaluation is skipped here
      if ((st.a - st.alpha) * st.fpa <= kDblEpsilon) { S3D_BFGS_HIT(kHitRoundoff); return bfgs_finish(st, kBfgsNoProgress, max_inner); }
      bfgs_set_trial(st); st.stage = kBfgsSection;
      return true;
    }
    // iteration caps reached: as in GSL / bfgs.h the step length is left as the caller initialised it (0); x0 + 0 p is x0, whose
    // value and gradient the state holds
    S3D_BFGS_HIT(kHitLineSearchCap);
    if (!bfgs_accept(st, 0.0, st.f, st.g0, max_inner)) return false;
    go = kGoStep;
  }
}

// f, g = objective at st.xc (the evaluation that was pending).  Returns true when another evaluation (at the new st.xc) is
// needed, false when the solve is over: result in st.x, st.failed set when PCL would reject it.
S3D_HD bool bfgs_advance(BfgsState& st, double f, const double (&g)[6], int max_inner) {
  const double f0 = st.f, fp0 = st.fp0;
  if (st.stage == kBfgsStart) {  // BFGS::minimizeInit
    st.delta_f = 0;
    st.f = f;
    for (int i = 0; i < 6; ++i) { st.x0[i] = st.x[i]; st.g0[i] = g[i]; }
    st.g0norm = bfgs_norm6(st.g0);
    for (int i = 0; i < 6; ++i) st.p[i] = g[i] * (-1.0 / st.g0norm);
    st.pnorm = bfgs_norm6(st.p);
    st.fp0 = -st.g0norm;
    return bfgs_run(st, kGoStep, max_inner);
  }
  const double falpha = f;
  if (st.stage == kBfgsBracket) {
    if (falpha > f0 + st.alpha * kBfgsRho * fp0 || falpha >= st.falpha_prev) {
      S3D_BFGS_HIT(kHitBracketRho);
      st.a = st.alpha_prev; st.fa = st.falpha_prev; st.fpa = st.fpalpha_prev;
      st.b = st.alpha; st.fb = falpha; st.fpb = NAN;
      return bfgs_run(st, kGoSection, max_inner);
    }
    const double fpalpha = bfgs_dot6(g, st.p);
    if (fabs(fpalpha) <= -kBfgsSigma * fp0) {
      S3D_BFGS_HIT(kHitBracketWolfe);
      return bfgs_accept(st, st.alpha, falpha, g, max_inner) && bfgs_run(st, kGoStep, max_inner);
    }
    if (fpalpha >= 0) {
      S3D_BFGS_HIT(kHitBracketSlope);
      st.a = st.alpha; st.fa = falpha; st.fpa = fpalpha;
      st.b = st.alpha_prev; st.fb = st.falpha_prev; st.fpb = st.fpalpha_prev;
      return bfgs_run(st, kGoSection, max_inner);
    }
    const double delta = st.alpha - st.alpha_prev;
    const double alpha_next = bfgs_interpolate(st.alpha_prev, st.falpha_prev, st.fpalpha_prev, st.alpha, falpha, fpalpha, st.alpha + delta,
                                               st.alpha + kBfgsTau1 * delta, kBfgsOrder);
    st.alpha_prev = st.alpha; st.falpha_prev = falpha; st.fpalpha_prev = fpalpha; st.alpha = alpha_next;
    return bfgs_run(st, kGoBracket, max_inner);
  }
  if (st.stage == kBfgsSection) {
    if (falpha > f0 + kBfgsRho * st.alpha * fp0 || falpha >= st.fa) {
      st.b = st.alpha; st.fb = falpha; st.fpb = NAN;
    } else {
      const double fpalpha = bfgs_dot6(g, st.p);
      if (fabs(fpalpha) <= -kBfgsSigma * fp0) {
        S3D_BFGS_HIT(kHitSectionWolfe);
        return bfgs_accept(st, st.alpha, falpha, g, max_inner) && bfgs_run(st, kGoStep, max_inner);
      }
      if (((st.b - st.a) >= 0 && fpalpha >= 0) || ((st.b - st.a) <= 0 && fpalpha <= 0)) { st.b = st.a; st.fb = st.fa; st.fpb = st.fpa; }
      st.a = st.alpha; st.fa = falpha; st.fpa = fpalpha;
    }
    return bfgs_run(st, kGoSection, max_inner);
  }
  return false;
}
}  // namespace s3d
