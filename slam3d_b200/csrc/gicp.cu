// gicp.cu — the Generalized-ICP loop of pcl::GeneralizedIterativeClosestPoint as driven by slam3d's doICP
// (slam3d/sensor/pcl/PointCloudSensor.cpp:52-82) and the fitness score of :73.   Semantics: SURVEY A.4-A.6.
//
// The whole loop of a batch is ONE persistent kernel (gicp_loop_kernel) with a device-side scheduler; the host launches it once
// and reads the results — no per-iteration launch, no host poll (round 1 spent 4 of 18 ms per 64 pairs in 690 control
// launches and 10 polls per chunk).  Pairs are independent, so there is no grid-wide barrier either: every pair is a small
// dataflow machine whose current PASS is published as (epoch, number of 256-point tiles); CTAs claim tiles of any pair with one
// atomic, and the CTA that delivers the last tile of a pass runs the pair's control step and publishes the next pass:
//   search pass   (iter_tile)     q = T_f32 * (guess_f32 * p) -> exact 1-NN in the fixed cloud (nn_search.cuh; skipped when the
//                                 previous correspondence is provably still nearest) -> d2 < max_corr^2 -> M = (R C1 R^T + C2)^-1
//                                 (FP64, stored) -> the 74 sums of gicp_math.h per tile in a fixed order: 60 x-independent sums
//                                 that give the whole Hessian, and the 13 residual sums + count of PCL's first objective evaluation
//   control step  (ctrl_step)     fixed-order sum of the tile partials, then ONE thread advances PCL's inner optimiser
//                                 (estimateRigidTransformationNewton, or per context the BFGS one of PCL <= 1.13, as a resumable
//                                 state machine, pair state staged in shared memory) to its next objective evaluation, or
//                                 finishes the outer iteration (convergence test)
//   trial pass    (eval_tile)     f (and its gradient) at the pending back-tracking / line-search trial(s): one pass over the stored correspondences with the
//                                 residual formed exactly as PCL forms it (float32 T(x)*p, float subtraction) -> 13 sums per tile
//   fitness pass  (fitness_tile)  getFitnessScore once the outer loop has ended; its last tile closes the pair
// While one pair sits in its (serial, ~10 us) control step the CTAs work on tiles of the other pairs; a CTA that finds nothing
// to claim sleeps (nanosleep) until a pass is published or no pair is active.  Progress never depends on a CTA that is not
// running: waiting CTAs wait only for tiles and control steps that are being executed.  A cycle-count watchdog ends the
// kernel with an error flag should that invariant ever be broken.
// Data written and read inside the kernel by different CTAs (pair state, correspondences, Mahalanobis matrices, search hints,
// tile partials) is handed over with a release atomic on the producer side and read from L2 (ld.global.cg) on the consumer
// side, because L1 is not coherent; the search structures (points, hash, normals) are immutable and stay on the cached path.
// (Tried and dropped, B200, 64 pairs per step: a separate search kernel in which one thread handles 2/3/4 consecutive points
// and passes each result on as a hint for the next — 10.1 / 11.6 / 13.0 ms per step against 8.6 ms; splitting the search and
// the 74-sum reduction into two kernels; per-lane cell cursors (+12 %); CTA-level compaction of the points that still need a
// search (equal): profiles/r01h_summary.md.  Round 2, first attempt: one launch per pass inside a CUDA-graph WHILE node with
// the control step fused by the same ticket scheme — correct, but every launch ended with one control step during which the
// GPU idled, and its __threadfence() calls dropped L1 once per tile: 13.3 ms per 64 pairs against 12.2 ms with separate
// control launches (profiles/r02_summary.md).)
// Because every float operation that PCL's decisions depend on is mirrored and the double sums differ only in order, the
// GPU follows the oracle's iterate sequence (same inner/outer iteration counts, bit-identical poses in the test-suite).
// Reductions use fixed trees: results are bit-reproducible run to run and independent of batch composition and scheduling.
// Roofline: per outer iteration 16 B (moving point) + 32 B (its normal) + gathered 16 B + 32 B (fixed point + normal) per
// correspondence, + 48 B (M) written; per evaluation 16 + 16 + 48 B.  The working set is L2 resident; the search is latency
// bound on the hash probes (DESIGN.md 4).
#include <cstdio>
#include <cstdlib>

#include "internal.h"
#include "nn_search.cuh"

namespace s3d {

constexpr int kFeat = 14;  // M00 M01 M02 M11 M12 M22 | px py pz | (Md)0 (Md)1 (Md)2 | d^T M d | valid

struct MomentSpec { uint8_t a, b, c; };  // moment = sum f[a]*f[b]*f[c]
struct SpecTable {                        // built at compile time: no per-device upload, nothing to race on
  MomentSpec s[kNumMoments];
  constexpr SpecTable() : s{} {
    const int phi[4] = {6, 7, 8, 13};
    int ab = 0;
    for (int a = 0; a < 3; ++a)
      for (int b = a; b < 3; ++b, ++ab) {
        int ce = 0;
        for (int c = 0; c < 4; ++c)
          for (int e = c; e < 4; ++e, ++ce) { s[ab * 10 + ce].a = (uint8_t)ab; s[ab * 10 + ce].b = (uint8_t)phi[c]; s[ab * 10 + ce].c = (uint8_t)phi[e]; }
      }
    for (int a = 0; a < 3; ++a) for (int c = 0; c < 4; ++c) { s[60 + a * 4 + c].a = (uint8_t)(9 + a); s[60 + a * 4 + c].b = (uint8_t)phi[c]; s[60 + a * 4 + c].c = 13; }
    s[72].a = 12; s[72].b = 13; s[72].c = 13;
    s[73].a = 13; s[73].b = 13; s[73].c = 13;
  }
};
__constant__ SpecTable c_spec = SpecTable();

// R = top-left 3x3 of double(T) * double(guess);  RRt = R R^T      (SURVEY A.4 "R <- ...")
__device__ void update_rotation(PairState& ps) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double s = 0;
      for (int k = 0; k < 4; ++k) s += (double)ps.T[k * 4 + i] * (double)ps.guess[j * 4 + k];
      ps.R[i][j] = s;
    }
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double s = 0;
      for (int k = 0; k < 3; ++k) s += ps.R[i][k] * ps.R[j][k];
      ps.RRt[i][j] = s;
    }
}

// Eigen Matrix4f * Matrix4f: ((a0*b0 + a1*b1) + a2*b2) + a3*b3, column-major
__device__ void mat4f_mul(const float* A, const float* B, float* C) {
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c)
      C[c * 4 + r] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(A[r], B[c * 4]), __fmul_rn(A[4 + r], B[c * 4 + 1])), __fmul_rn(A[8 + r], B[c * 4 + 2])),
                               __fmul_rn(A[12 + r], B[c * 4 + 3]));
}

__device__ __noinline__ void bfgs_begin_outer(PairState& ps) {  // out of line: the Newton path does not carry it
  bfgs_begin(ps.bst, ps.T);
  matrix_from_state(ps.bst.xc, ps.T_eval);
}

// start of an outer iteration: x0 from transformation_, the float matrix PCL's first evaluation uses, and R for the Mahalanobis matrices
__device__ void begin_outer(PairState& ps) {
  if (ps.optimizer == S3D_GICP_BFGS) {
    bfgs_begin_outer(ps);
  } else {
    newton_begin(ps.nst, ps.T);
    matrix_from_state(ps.nst.xc, ps.T_eval);
  }
  update_rotation(ps);
  ps.phase = kPhaseNeedNN;
}

// Registration::align set-up: gates of align() :134-135, output = guess * input (transformPointCloud), state reset.
__global__ void __launch_bounds__(256) gicp_prepare_kernel(const SlotInfo* __restrict__ slots, PairState* __restrict__ pairs,
                                                           float4* __restrict__ moved, uint32_t* __restrict__ prev_nn, float* __restrict__ sec_lb,
                                                           PairSched* __restrict__ psched, int32_t* __restrict__ flags) {
  const uint32_t p = blockIdx.y;
  PairState& ps = pairs[p];
  const SlotInfo& sb = slots[2 * p];      // fixed cloud B  (slam3d source = PCL target)
  const SlotInfo& sa = slots[2 * p + 1];  // moving cloud A (slam3d target = PCL source)
  const bool enough = sa.n_pts >= 100 && sb.n_pts >= 100;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    ps.active = enough ? 1 : 0;
    ps.phase = kPhaseFinished;
    ps.ticket = 0;
    if (enough) { begin_outer(ps); atomicAdd(&flags[1], 1); }
    // first pass (epoch 1): the search pass of outer iteration 1, or nothing for a pair that fails the <100-point gate
    psched[p].desc = (1ull << 32) | (enough ? (1u << 24) | ((sa.n_pts + kIterTile - 1) / kIterTile) : 0u);
    psched[p].claim = 1ull << 32;
  }
  if (!enough) return;
  for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < sa.n_pts; r += gridDim.x * blockDim.x) {  // any grid covers the cloud (Workspace::grid_frac)
    const float4 v = sa.gpts[r];
    const float3 m = transform_se3(ps.guess, v.x, v.y, v.z);
    moved[ps.pt_off + r] = make_float4(m.x, m.y, m.z, v.w);
    prev_nn[ps.pt_off + r] = kNoIndex;
    sec_lb[ps.pt_off + r] = 0.f;
  }
}

// Temporal-coherence certificate (exactness preserving).  The last search for this point ran at position q_old and left
// (j, lb): every fixed point other than j was at least `lb` away from q_old.  If the query moved by m and
// dist(q_new, p_j) < lb - m, then j is still the unique nearest neighbour at q_new and no search is needed; the bound for
// the next iteration becomes lb - m.  Generous relative slack (1e-5) covers the float rounding of dist2_pcl (4e-7).
__device__ __forceinline__ bool certified_same_nn(const GridView& g, float3 q, float3 q_old, uint32_t j, float lb, NNResult& nn, float& lb_new) {
  if (j >= g.n || !(lb > 0.f)) return false;
  const float mx = q.x - q_old.x, my = q.y - q_old.y, mz = q.z - q_old.z;
  const float m = sqrtf(mx * mx + my * my + mz * mz) * 1.00001f + 1e-7f;
  const float rest = (lb - m) * 0.99999f;
  if (!(rest > 0.f)) return false;
  const float4 v = __ldg(g.pts + j);
  const float d2 = dist2_pcl(q.x, q.y, q.z, v.x, v.y, v.z);
  if (!(d2 * 1.00001f < rest * rest)) return false;
  nn.d2 = d2; nn.idx = __float_as_uint(v.w); nn.pos = j; nn.lb2 = rest * rest;
  lb_new = rest;
  return true;
}

// ---- shared-memory plan of gicp_loop_kernel ---------------------------------------------------------------------------------
// [0, kSmTile)  tile scratch.  search pass: feat[256][14] | part[3][74] | noted cells;  trial pass: feat[256][8] | part[16][13];
//                fitness pass: sums[256] | counts[256] | ... | noted cells;  control step: CtrlShared from 0.
// The read-only copy of the pair state of the tile being processed (fetched from L2) sits in a part of the scratch that its
// pass does not touch while the state is read: at kSmStateA (inside the feat area, which the search and fitness passes only
// write after their searches — behind a barrier) or at kSmStateB (the noted-cells area, unused by the trial pass).
// 46 832 B per CTA keeps four CTAs per SM inside the 196 KB shared-memory carve-out, i.e. 60 KB of L1 for the searches; a
// separate 2.5 KB slot for the pair state pushed the carve-out to 228 KB and halved L1 (measured: profiles/r02_summary.md).
constexpr size_t kSmPart = size_t(kIterTile) * kFeat * 8;                  // after feat[256][14]
constexpr size_t kSmCells = kSmPart + 3 * kNumMoments * 8;                  // after part[3][74]
constexpr size_t kSmTile = kSmCells + size_t(kNNGatherCap) * kIterTile * 8; // 46 832 B
constexpr size_t kSmLoop = kSmTile;
constexpr size_t kSmStateA = 4096, kSmStateB = kSmCells;
static_assert(kSmStateA >= size_t(kIterTile) * 12 && kSmStateA + sizeof(PairState) <= kSmPart, "pair state vs fitness sums / feat area");
static_assert(kSmStateB >= size_t(kIterTile) * 64 + 16 * kEvalSums * 8 && kSmStateB + sizeof(PairState) <= kSmTile, "pair state vs trial-pass scratch");

__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p) { return *reinterpret_cast<const volatile unsigned long long*>(p); }
__device__ __forceinline__ int32_t ld_volatile_i32(const int32_t* p) { return *reinterpret_cast<const volatile int32_t*>(p); }
__device__ __forceinline__ unsigned long long global_ns() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ uint32_t sm_id() { uint32_t r; asm volatile("mov.u32 %0, %%smid;" : "=r"(r)); return r; }
// Release-only operations (MEMBAR.ALL.GPU + the atomic).  __threadfence() and every acquire form additionally emit CCTL.IVALL,
// which drops the SM's whole L1 — the cache the searches of all resident CTAs live on — so the consumer side of every hand-over
// in this kernel is a relaxed atomic followed by L2 loads (ld.global.cg / volatile) whose addresses depend on its result.
__device__ __forceinline__ uint32_t atom_add_release(uint32_t* p, uint32_t v) {
  uint32_t old;
  asm volatile("atom.add.release.gpu.global.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ void exch_release(unsigned long long* p, unsigned long long v) {
  unsigned long long old;
  asm volatile("atom.exch.release.gpu.global.b64 %0, [%1], %2;" : "=l"(old) : "l"(p), "l"(v) : "memory");
  (void)old;
}
__device__ __forceinline__ void red_add_release(int32_t* p, int32_t v) { asm volatile("red.add.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }

// kShared = true: called from the persistent kernel — the pair state is a copy inside the scratch, and data written by other CTAs
// of the same launch is read from L2.  kShared = false: called from a per-pass kernel — the pair state is read in place and
// everything written before the launch is visible through L1.
template <bool kShared, typename T>
__device__ __forceinline__ T ld_pass(const T* p) { return kShared ? __ldcg(p) : *p; }

__device__ __forceinline__ double4 ldg_normal(const double4* p) {  // unit normal (x, y, z) through the read-only path; .w is padding
  const double2 xy = __ldg(reinterpret_cast<const double2*>(p));
  return make_double4(xy.x, xy.y, __ldg(reinterpret_cast<const double*>(p) + 2), 0.0);
}

// search pass of one tile
template <bool kShared>
__device__ __forceinline__ void iter_tile(const GicpArgs& a, const PairState& ps, const SlotInfo& sb, const SlotInfo& sa, uint32_t p, uint32_t tile,
                                          unsigned char* smem) {
  double (*feat)[kFeat] = reinterpret_cast<double (*)[kFeat]>(smem);
  double (*part)[kNumMoments] = reinterpret_cast<double (*)[kNumMoments]>(smem + kSmPart);
  uint2* s_cells = reinterpret_cast<uint2*>(smem + kSmCells);  // cell ranges noted by the gathering search (nn_search.cuh)
  const uint32_t r = tile * kIterTile + threadIdx.x;
  double f[kFeat];
#pragma unroll
  for (int i = 0; i < kFeat; ++i) f[i] = 0.0;
  if (r < sa.n_pts) {
    const GridView g = make_grid_view(sb);
    const float4 mv = __ldg(a.moved + ps.pt_off + r);  // moved[], the normals and the sorted points never change during the loop: read-only path
    const float3 q = transform_mv(ps.T, mv.x, mv.y, mv.z);
    const double thr = ps.max_corr2;
    const float cutoff = __double2float_ru(thr);
    const uint32_t hint = ld_pass<kShared>(a.prev_nn + ps.pt_off + r);  // written by the previous search pass, possibly on another SM
    NNResult nn;
    float lb_new;
    if (!certified_same_nn(g, q, transform_mv(ps.T_search, mv.x, mv.y, mv.z), hint, ld_pass<kShared>(a.sec_lb + ps.pt_off + r), nn, lb_new)) {
      nn = nn_search<true>(g, q.x, q.y, q.z, cutoff, hint, kNoIndex, s_cells + threadIdx.x);
      a.prev_nn[ps.pt_off + r] = nn.pos;
      lb_new = sqrtf(nn.lb2) * 0.99999f;
    }
    a.sec_lb[ps.pt_off + r] = lb_new;
    uint32_t c = kNoIndex;
    if (nn.pos != kNoIndex && (double)nn.d2 < thr) {
      c = nn.pos;
      const double4 n1 = ldg_normal(sa.normals + r);
      const double4 n2 = ldg_normal(sb.normals + nn.pos);
      double av[3], bv[3] = {n2.x, n2.y, n2.z};
      for (int i = 0; i < 3; ++i) av[i] = ps.R[i][0] * n1.x + ps.R[i][1] * n1.y + ps.R[i][2] * n1.z;
      double M[6];
      mahalanobis6(ps.RRt, av, bv, M);
      double* mo = a.mahal + 6 * (size_t)(ps.pt_off + r);
#pragma unroll
      for (int i = 0; i < 6; ++i) mo[i] = M[i];
      // PCL's first objective evaluation of this outer iteration: d = float(T(x0) * p) - q, float subtraction, then double
      const float4 qb = __ldg(g.pts + nn.pos);
      const float3 pp = transform_mv(ps.T_eval, mv.x, mv.y, mv.z);
      const double d0 = (double)__fsub_rn(pp.x, qb.x), d1 = (double)__fsub_rn(pp.y, qb.y), d2 = (double)__fsub_rn(pp.z, qb.z);
      const double Md0 = M[0] * d0 + M[1] * d1 + M[2] * d2;
      const double Md1 = M[1] * d0 + M[3] * d1 + M[4] * d2;
      const double Md2 = M[2] * d0 + M[4] * d1 + M[5] * d2;
#pragma unroll
      for (int i = 0; i < 6; ++i) f[i] = M[i];
      f[6] = mv.x; f[7] = mv.y; f[8] = mv.z;
      f[9] = Md0; f[10] = Md1; f[11] = Md2;
      f[12] = d0 * Md0 + d1 * Md1 + d2 * Md2;
      f[13] = 1.0;
    }
    a.corr[ps.pt_off + r] = c;
  }
  if (kShared) __syncthreads();  // every thread is done with the pair state, which lives inside the feat area
#pragma unroll
  for (int i = 0; i < kFeat; ++i) feat[threadIdx.x][i] = f[i];
  __syncthreads();
  // 74 sums x 3 sub-ranges of the tile, each summed in ascending point order
  if (threadIdx.x < 3 * kNumMoments) {
    const int m = threadIdx.x % kNumMoments, sub = threadIdx.x / kNumMoments;
    const MomentSpec sp = c_spec.s[m];
    const int lo = sub * 86, hi = min(kIterTile, lo + 86);
    double s = 0.0;
    for (int i = lo; i < hi; ++i) s += feat[i][sp.a] * feat[i][sp.b] * feat[i][sp.c];
    part[sub][m] = s;
  }
  __syncthreads();
  if (threadIdx.x < kNumMoments) {
    const size_t t = (size_t)p * a.tiles_per_pair + tile;
    a.moments[t * kNumMoments + threadIdx.x] = (part[0][threadIdx.x] + part[1][threadIdx.x]) + part[2][threadIdx.x];
  }
}

// trial pass of one tile: 13 residual sums per pending back-tracking trial, residual formed exactly as PCL forms it
template <bool kShared>
__device__ __forceinline__ void eval_tile(const GicpArgs& a, const PairState& ps, const SlotInfo& sb, const SlotInfo& sa, uint32_t p, uint32_t tile,
                                          unsigned char* smem) {
  double (*feat)[8] = reinterpret_cast<double (*)[8]>(smem);                                   // px py pz | (Md)0..2 | d^T M d | 1
  double (*part)[kEvalSums] = reinterpret_cast<double (*)[kEvalSums]>(smem + size_t(kIterTile) * 8 * 8);
  const uint32_t r = tile * kIterTile + threadIdx.x;
  bool valid = false;
  float4 mv = make_float4(0.f, 0.f, 0.f, 0.f), qb = mv;
  double M[6] = {0, 0, 0, 0, 0, 0};
  if (r < sa.n_pts) {
    const uint32_t c = ld_pass<kShared>(a.corr + ps.pt_off + r);  // written by the search pass, possibly on another SM
    if (c != kNoIndex) {
      valid = true;
      mv = __ldg(a.moved + ps.pt_off + r);
      qb = __ldg(sb.gpts + c);
      const double* Mp = a.mahal + 6 * (size_t)(ps.pt_off + r);
#pragma unroll
      for (int i = 0; i < 6; ++i) M[i] = ld_pass<kShared>(Mp + i);
    }
  }
  const size_t t = (size_t)p * a.tiles_per_pair + tile;
  const int j0 = ps.trial_first, j1 = ps.trial_first + ps.trial_count;
  for (int j = j0; j < j1; ++j) {
    double f[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (valid) {
      const float3 pp = transform_mv(ps.T_trial[j], mv.x, mv.y, mv.z);
      const double d0 = (double)__fsub_rn(pp.x, qb.x), d1 = (double)__fsub_rn(pp.y, qb.y), d2 = (double)__fsub_rn(pp.z, qb.z);
      const double Md0 = M[0] * d0 + M[1] * d1 + M[2] * d2;
      const double Md1 = M[1] * d0 + M[3] * d1 + M[4] * d2;
      const double Md2 = M[2] * d0 + M[4] * d1 + M[5] * d2;
      f[0] = mv.x; f[1] = mv.y; f[2] = mv.z; f[3] = Md0; f[4] = Md1; f[5] = Md2;
      f[6] = d0 * Md0 + d1 * Md1 + d2 * Md2; f[7] = 1.0;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) feat[threadIdx.x][i] = f[i];
    __syncthreads();
    // sum s (0..11: (Md)_a * phi_c with a = s / 4, c = s % 4; 12: d^T M d) over 16 sub-ranges of 16 points, ascending order
    if (threadIdx.x < 16 * kEvalSums) {
      const int sidx = threadIdx.x % kEvalSums, sub = threadIdx.x / kEvalSums;
      const int ia = sidx < 12 ? 3 + sidx / 4 : 6;
      const int ib = sidx < 12 ? (sidx % 4 < 3 ? sidx % 4 : 7) : 7;
      double acc = 0.0;
      for (int i = sub * 16; i < sub * 16 + 16; ++i) acc += feat[i][ia] * feat[i][ib];
      part[sub][sidx] = acc;
    }
    __syncthreads();
    if (threadIdx.x < kEvalSums) {
      double acc = 0.0;
      for (int sub = 0; sub < 16; ++sub) acc += part[sub][threadIdx.x];
      a.eval_part[(t * kLineSearchTrials + j) * kEvalSums + threadIdx.x] = acc;
    }
  }
}

// fitness pass of one tile — getFitnessScore(max_range): transformPointCloud(input, final), 1-NN, d2 <= max_range (sic), mean of d2 (A.6)
template <bool kShared>
__device__ __forceinline__ void fitness_tile(const GicpArgs& a, const PairState& ps, const SlotInfo& sb, const SlotInfo& sa, uint32_t p, uint32_t tile,
                                             unsigned char* smem) {
  double* ssum = reinterpret_cast<double*>(smem);
  uint32_t* scnt = reinterpret_cast<uint32_t*>(smem + size_t(kIterTile) * 8);
  uint2* s_cells = reinterpret_cast<uint2*>(smem + kSmCells);
  const uint32_t r = tile * kIterTile + threadIdx.x;
  double s = 0.0; uint32_t c = 0;
  if (r < sa.n_pts) {
    const GridView g = make_grid_view(sb);
    const float4 v = __ldg(sa.gpts + r);
    const float3 q = transform_se3(ps.final_T, v.x, v.y, v.z);
    const float4 mv = __ldg(a.moved + ps.pt_off + r);
    const uint32_t hint = ld_pass<kShared>(a.prev_nn + ps.pt_off + r);
    NNResult nn;
    float lb_new;
    if (!certified_same_nn(g, q, transform_mv(ps.T_search, mv.x, mv.y, mv.z), hint, ld_pass<kShared>(a.sec_lb + ps.pt_off + r), nn, lb_new))
      nn = nn_search<true>(g, q.x, q.y, q.z, __double2float_ru(ps.fit_range), hint, kNoIndex, s_cells + threadIdx.x);
    if (nn.pos != kNoIndex && (double)nn.d2 <= ps.fit_range) { s = (double)nn.d2; c = 1; }
  }
  ssum[threadIdx.x] = s; scnt[threadIdx.x] = c;  // [0, 3072): below the pair state at kSmStateA
  __syncthreads();
  for (int o = kIterTile / 2; o > 0; o >>= 1) {  // fixed tree
    if (threadIdx.x < o) { ssum[threadIdx.x] += ssum[threadIdx.x + o]; scnt[threadIdx.x] += scnt[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const size_t t = (size_t)p * a.tiles_per_pair + tile;
    a.fit_partial[2 * t] = ssum[0];
    a.fit_partial[2 * t + 1] = (double)scnt[0];
  }
}

// End of an outer iteration (computeTransformation, SURVEY A.4): convergence test, counters, next iteration or final transform.
// x, inner: the inner optimiser's result state and iteration count.
__device__ void finish_outer(PairState& ps, bool optimiser_failed, const double* x, int inner) {
  bool stop = false;
  if (optimiser_failed) {
    ps.failed = 1; ps.converged = 0; stop = true;  // optimiser exception: loop breaks, converged_ stays false, final = previous * guess
  } else {
    float T[16];
    matrix_from_state(x, T);  // transformation_matrix.setIdentity(); applyState(transformation_matrix, x)
    ps.inner_iterations += inner;
    double delta = 0.0;
    for (int r = 0; r < 4; ++r)
      for (int c = 0; c < 4; ++c) {
        const double ratio = (r < 3 && c < 3) ? 1.0 / ps.rot_eps : 1.0 / ps.trans_eps;
        const double cd = ratio * fabs((double)ps.prev[c * 4 + r] - (double)T[c * 4 + r]);
        if (cd > delta) delta = cd;
      }
    for (int i = 0; i < 16; ++i) ps.T[i] = T[i];
    ps.outer_iterations += 1;
    if (ps.outer_iterations >= ps.max_iter || delta < 1.0) {
      ps.converged = 1; stop = true;
      for (int i = 0; i < 16; ++i) ps.prev[i] = T[i];  // previous_transformation_ = transformation_
    }
  }
  if (stop) {
    mat4f_mul(ps.prev, ps.guess, ps.final_T);  // final_transformation_ = previous_transformation_ * guess
    ps.phase = kPhaseFitness;                  // the pair stays active until its fitness pass has been summed
  } else {
    begin_outer(ps);
  }
}

// euler_derivs(x, E, true) spread over the CTA: threads 0..2 build the factor matrices of one axis each (the three sincos),
// threads 0..9 one product (A B) C each, with the same operand order as the serial function, so E is bit-identical.
__device__ void euler_derivs_cta(const double* x, Euler& E, double (*fac)[3][3][3]) {  // fac[axis][order] in shared memory
  const int t = threadIdx.x;
  if (t < 3) euler_factor(x[3 + t], t, fac[t][0], fac[t][1], fac[t][2]);  // axis 0 = X(phi), 1 = Y(theta), 2 = Z(psi)
  __syncthreads();
  if (t < 10) {
    // derivative orders (z, y, x) of: R | dR0 dR1 dR2 | ddR00 ddR11 ddR22 | ddR01 ddR02 ddR12
    const int oz = (t == 3) ? 1 : (t == 6) ? 2 : (t == 8 || t == 9) ? 1 : 0;
    const int oy = (t == 2) ? 1 : (t == 5) ? 2 : (t == 7 || t == 9) ? 1 : 0;
    const int ox = (t == 1) ? 1 : (t == 4) ? 2 : (t == 7 || t == 8) ? 1 : 0;
    double T[3][3], O[3][3];
    mat3_mul(fac[2][oz], fac[1][oy], T);
    mat3_mul(T, fac[0][ox], O);
    double (*dst)[3] = t == 0 ? E.R : t == 1 ? E.dR[0] : t == 2 ? E.dR[1] : t == 3 ? E.dR[2] : t == 4 ? E.ddR[0][0] : t == 5 ? E.ddR[1][1]
                     : t == 6 ? E.ddR[2][2] : t == 7 ? E.ddR[0][1] : t == 8 ? E.ddR[0][2] : E.ddR[1][2];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) dst[i][j] = O[i][j];
    if (t >= 7) {  // mixed second derivatives are symmetric in (k, l)
      double (*sym)[3] = t == 7 ? E.ddR[1][0] : t == 8 ? E.ddR[2][0] : E.ddR[2][1];
      for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) sym[i][j] = O[i][j];
    }
  }
  __syncthreads();
}

// Control step of pair p, run by the CTA that delivered the last tile of a search or trial pass: ordered reduction of the tile
// partials, then the optimiser advances.  The pair state is staged in shared memory (the serial part is one thread's dependent
// chain; on global memory every step of it was an L2 round trip: 29 us per control launch in round 1).
// BFGS mode (PCL <= 1.13): f and the gradient at the pending state (sums 60..73, gradient entries gH[0..5]) advance the line
// search to its next trial, which becomes the single trial T_trial[0] of the next pass, or end the solve.  Out of line: the
// Newton path of the loop kernel does not carry its registers.
__device__ __noinline__ void bfgs_ctrl(PairState& ps, const double* gH) {
  double g[6];
  for (int i = 0; i < 6; ++i) g[i] = gH[i];
  if (bfgs_advance(ps.bst, ps.sums[72] / ps.sums[73], g, ps.max_inner)) {
    matrix_from_state(ps.bst.xc, ps.T_trial[0]);
    ps.trial_first = 0; ps.trial_count = 1;
    ps.phase = kPhaseEval;
  } else {
    if (ps.bst.failed) ps.inner_iterations += ps.bst.it;  // estimateRigidTransformationBFGS has counted them before it throws
    finish_outer(ps, ps.bst.failed != 0, ps.bst.x, ps.bst.it);
  }
}

struct CtrlShared {
  PairState ps;
  double part[3][kLineSearchTrials * kEvalSums];
  double red[kLineSearchTrials * kEvalSums];
  Euler E;
  double fac[3][3][3][3];
  double gH[42];
  int mode;      // 0: nothing to assemble, 1: assemble the objective at ps.nst.xc from ps.sums
  int newstep;   // a new Newton step started: its trial matrices are needed
};
static_assert(sizeof(CtrlShared) <= kSmTile, "control step must fit into the tile scratch");

__device__ __forceinline__ void ctrl_step_body(const GicpArgs& a, uint32_t p, int after_eval, unsigned char* smem) {
  CtrlShared& sh = *reinterpret_cast<CtrlShared*>(smem);
  PairState& ps = sh.ps;
  PairState* psg = a.pairs + p;
  {
    const unsigned long long* src = reinterpret_cast<const unsigned long long*>(psg);
    unsigned long long* dst = reinterpret_cast<unsigned long long*>(&sh.ps);
    for (uint32_t i = threadIdx.x; i < sizeof(PairState) / 8; i += blockDim.x) dst[i] = __ldcg(src + i);
  }
  __syncthreads();
  const uint32_t n_tiles = (a.slots[2 * p + 1].n_pts + kIterTile - 1) / kIterTile;
  const int n_sums = after_eval ? ps.trial_count * kEvalSums : kNumMoments;
  const int stride = after_eval ? kLineSearchTrials * kEvalSums : kNumMoments;
  const double* src0 = after_eval ? a.eval_part + (size_t)p * a.tiles_per_pair * stride + ps.trial_first * kEvalSums
                                  : a.moments + (size_t)p * a.tiles_per_pair * stride;
  // fixed order: `subs` contiguous tile ranges per sum, each summed front to back, then the ranges front to back.  As many ranges
  // as the CTA has threads for (3 for the 74 sums of a search pass, 16 for the 13 of a single trial): the chain of dependent L2
  // loads per thread is what this step waits for.
  const int subs = min(16, 256 / n_sums);
  double* part = &sh.part[0][0];  // [subs][n_sums], at most 3 * 130 entries
  if ((int)threadIdx.x < subs * n_sums) {
    const int m = threadIdx.x % n_sums, sub = threadIdx.x / n_sums;
    const uint32_t per = (n_tiles + subs - 1) / subs;
    const uint32_t lo = sub * per, hi = min(n_tiles, lo + per);
    const double* src = src0 + m;
    double s = 0.0;
#pragma unroll 8
    for (uint32_t t = lo; t < hi; ++t) s += __ldcg(src + (size_t)t * stride);  // written by other CTAs: read from L2
    part[sub * n_sums + m] = s;
  }
  __syncthreads();
  if ((int)threadIdx.x < n_sums) {
    double s = part[threadIdx.x];
    for (int sub = 1; sub < subs; ++sub) s += part[sub * n_sums + threadIdx.x];
    sh.red[threadIdx.x] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    sh.mode = 1; sh.newstep = 0;
    ps.ticket = 0;
    if (!after_eval) {
      for (int i = 0; i < kNumMoments; ++i) ps.sums[i] = sh.red[i];
      ps.n_corr = (uint32_t)ps.sums[73];
      for (int i = 0; i < 16; ++i) { ps.prev[i] = ps.T[i]; ps.T_search[i] = ps.T[i]; }  // previous_transformation_ = transformation_
      if (ps.sums[73] < 4.0) { finish_outer(ps, true, ps.nst.x, 0); sh.mode = 0; }  // min_number_correspondences_: PCL throws
    } else if (ps.optimizer == S3D_GICP_BFGS) {
      for (int i = 0; i < kEvalSums; ++i) ps.sums[60 + i] = sh.red[i];  // the single pending line-search trial
    } else {
      double f_trial[kLineSearchTrials];
      for (int j = 0; j < ps.trial_count; ++j) f_trial[ps.trial_first + j] = sh.red[j * kEvalSums + 12] / ps.sums[73];
      const int j = newton_pick_trial(ps.nst, f_trial, ps.trial_first, ps.trial_count);
      if (j >= 0) {
        newton_select_trial(ps.nst, j);
        for (int i = 0; i < kEvalSums; ++i) ps.sums[60 + i] = sh.red[(j - ps.trial_first) * kEvalSums + i];
      } else if (ps.trial_first == 0 && kLineSearchTrials > 1) {
        ps.trial_first = 1; ps.trial_count = kLineSearchTrials - 1;  // trial 0 did not improve: evaluate all remaining trials in one pass
        sh.mode = 0;
      } else {
        ps.nst.phase = 2;  // no improvement found
        finish_outer(ps, false, ps.nst.x, ps.nst.it);
        sh.mode = 0;
      }
    }
  }
  __syncthreads();
  if (sh.mode) {
    euler_derivs_cta(ps.optimizer == S3D_GICP_BFGS ? ps.bst.xc : ps.nst.xc, sh.E, sh.fac);
    // objective at the evaluated state: 42 threads contract one gradient / Hessian entry each
    if (threadIdx.x < 42) sh.gH[threadIdx.x] = objective_entry(ps.sums, sh.E, threadIdx.x);
    __syncthreads();
    if (threadIdx.x == 0 && ps.optimizer == S3D_GICP_BFGS) {
      bfgs_ctrl(ps, sh.gH);
    } else if (threadIdx.x == 0) {
      double g[6], H[6][6];
      for (int i = 0; i < 6; ++i) { g[i] = sh.gH[i]; for (int j = 0; j < 6; ++j) H[i][j] = sh.gH[6 + 6 * i + j]; }
      if (newton_advance_pre(ps.nst, ps.sums[72] / ps.sums[73], g, H, ps.max_inner)) {
        ps.trial_first = 0; ps.trial_count = 1;
        ps.phase = kPhaseEval;
        sh.newstep = 1;
      } else {
        finish_outer(ps, false, ps.nst.x, ps.nst.it);
      }
    }
    __syncthreads();
    if (sh.newstep && threadIdx.x < kLineSearchTrials) {  // float matrices of all back-tracking trials of the new step
      double xc[6];
      newton_trial_state(ps.nst, threadIdx.x, xc);
      matrix_from_state(xc, ps.T_trial[threadIdx.x]);
    }
  }
  __syncthreads();
  {
    const unsigned long long* src = reinterpret_cast<const unsigned long long*>(&sh.ps);
    unsigned long long* dst = reinterpret_cast<unsigned long long*>(psg);
    for (uint32_t i = threadIdx.x; i < sizeof(PairState) / 8; i += blockDim.x) dst[i] = src[i];
  }
}

// last tile of the fitness pass: ordered sum of the tile partials (same order as a sequential loop over the tiles); closes the pair
__device__ void fitness_finish(const GicpArgs& a, uint32_t p, unsigned char* smem) {
  double* part = reinterpret_cast<double*>(smem);
  const uint32_t n_tiles = (a.slots[2 * p + 1].n_pts + kIterTile - 1) / kIterTile;
  const double* src = a.fit_partial + 2 * (size_t)p * a.tiles_per_pair;
  double s = 0.0, c = 0.0;
  for (uint32_t base = 0; base < n_tiles; base += kIterTile) {  // 256 tiles at a time through shared memory
    const uint32_t t = base + threadIdx.x;
    if (t < n_tiles) { part[2 * threadIdx.x] = __ldcg(src + 2 * t); part[2 * threadIdx.x + 1] = __ldcg(src + 2 * t + 1); }
    __syncthreads();
    if (threadIdx.x == 0) {
      const uint32_t m = min((uint32_t)kIterTile, n_tiles - base);
      for (uint32_t i = 0; i < m; ++i) { s += part[2 * i]; c += part[2 * i + 1]; }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    PairState* psg = a.pairs + p;
    psg->fit_sum = s; psg->fit_n = (uint32_t)c;
    psg->ticket = 0;
    psg->phase = kPhaseFinished;
    psg->active = 0;
  }
}

// cooperative copy of the pair state from L2 into shared memory (explicitly global loads: every field a tile reads afterwards is
// an LDS broadcast instead of a generic load per thread)
__device__ __forceinline__ const PairState& stage_state(const GicpArgs& a, uint32_t p, unsigned char* dst) {
  const unsigned long long* src = reinterpret_cast<const unsigned long long*>(a.pairs + p);
  unsigned long long* d = reinterpret_cast<unsigned long long*>(dst);
  for (uint32_t i = threadIdx.x; i < sizeof(PairState) / 8; i += blockDim.x) d[i] = __ldcg(src + i);
  __syncthreads();
  return *reinterpret_cast<const PairState*>(dst);
}

// ---- scheduler ------------------------------------------------------------------------------------------------------------------
// PairSched.desc  = epoch << 32 | tiles per claim << 24 | tiles of the pass that is open for claims (0 tiles: nothing to claim —
//                   control step running, or the pair is closed)
// PairSched.claim = epoch << 32 | next unclaimed tile.  A pass is published by writing desc first and claim second, so whoever
// draws (epoch, t) from `claim` finds the descriptor of that epoch; claims past the end of a pass are harmless.
// The first warp of a CTA claims: its lanes look at 32 pairs at once (two loads per lane, one L2 round trip for the warp), the
// candidate nearest to the pair the CTA worked on last draws with one atomic — n tiles at a time (1 for the search and fitness
// passes, kTrialTilesPerClaim for the cheap trial passes, whose fixed cost per claim — state fetch, ticket, barriers — would
// otherwise match their work).
constexpr uint32_t kTrialTilesPerClaim = 4;
constexpr uint32_t kAvailMask = 0x00FFFFFFu;

__device__ __forceinline__ bool claim_tiles_warp(const GicpArgs& a, uint32_t& rot, uint32_t& p_out, uint32_t& t_out, uint32_t& n_out) {
  const uint32_t FULL = 0xFFFFFFFFu;
  const uint32_t lane = threadIdx.x & 31u;
  for (uint32_t base = 0; base < a.n_pairs; base += 32) {
    const bool in = base + lane < a.n_pairs;
    uint32_t p = rot + base + lane;
    if (p >= a.n_pairs) p -= a.n_pairs;
    unsigned long long d = 0, c = 0;
    if (in) { d = ld_volatile_u64(&a.psched[p].desc); c = ld_volatile_u64(&a.psched[p].claim); }
    const uint32_t per = max(1u, (uint32_t)d >> 24);
    const bool cand = in && ((uint32_t)d & kAvailMask) != 0u && (c >> 32) == (d >> 32) && (uint32_t)c < ((uint32_t)d & kAvailMask);
    uint32_t m = __ballot_sync(FULL, cand);
    while (m) {
      const int src = __ffs(m) - 1;
      m &= m - 1;
      unsigned long long cc = 0, dd = d;
      if ((int)lane == src) {
        cc = atomicAdd(&a.psched[p].claim, (unsigned long long)per);
        if ((cc >> 32) != (d >> 32)) dd = ld_volatile_u64(&a.psched[p].desc);  // drawn from a newer pass: its descriptor is already published
      }
      cc = __shfl_sync(FULL, cc, src); dd = __shfl_sync(FULL, dd, src);
      const uint32_t pp = __shfl_sync(FULL, p, src), added = __shfl_sync(FULL, per, src);
      const uint32_t avail = (uint32_t)dd & kAvailMask, t0 = (uint32_t)cc;
      if ((cc >> 32) == (dd >> 32) && t0 < avail) { rot = pp; p_out = pp; t_out = t0; n_out = min(added, avail - t0); return true; }
    }
  }
  return false;
}

__device__ __forceinline__ void publish_pass(const GicpArgs& a, uint32_t p, uint32_t n_tiles, uint32_t per_claim) {
  PairSched* s = a.psched + p;
  const unsigned long long epoch = (ld_volatile_u64(&s->desc) >> 32) + 1ull;
  exch_release(&s->desc, (epoch << 32) | (n_tiles ? (per_claim << 24) | n_tiles : 0u));  // release: the pair state written by this CTA comes first
  if (n_tiles) exch_release(&s->claim, epoch << 32);                                      // release: the descriptor comes before its claims
}

// LATENCY mode — single registrations and small batches, one call at a time: the whole loop in ONE launch.  A CTA that finds
// nothing to claim waits (nanosleep) for the next pass to be published.  Two CTAs per SM (128 registers): a single pair has 185
// tiles per pass for 148 SMs, so occupancy is not what limits it — the serial control step is, and with 128 registers it runs
// without the spills a 64-register budget forces on its FP64 chain.
__global__ void __launch_bounds__(kIterTile, 2) gicp_loop_kernel(const __grid_constant__ GicpArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ uint32_t s_p, s_tile, s_n;
  __shared__ int s_found, s_last;
  uint32_t rot = sm_id() % a.n_pairs;  // the CTAs of one SM start on the same pair: its grid and points share that SM's L1
  const long long t_start = clock64();
  for (;;) {
    if (threadIdx.x < 32) {  // the first warp looks for work; the others wait at the barrier
      int found = 0;
      uint32_t cp = 0, ct = 0, cn = 0;
      for (uint32_t spin = 0;; ++spin) {
        if (claim_tiles_warp(a, rot, cp, ct, cn)) { found = 1; break; }
        if (ld_volatile_i32(&a.flags[1]) <= 0 || (ld_volatile_i32(&a.flags[0]) & kErrWatchdog)) break;  // no pair is active: done
        __nanosleep(spin < 8 ? 100 : 400);
        if ((spin & 255u) == 255u && clock64() - t_start > (long long)a.watchdog_cycles) { atomicOr(&a.flags[0], kErrWatchdog); break; }
      }
      if (threadIdx.x == 0) { s_found = found; s_p = cp; s_tile = ct; s_n = cn; }
    }
    __syncthreads();
    if (!s_found) break;
    const uint32_t p = s_p, tile0 = s_tile, n_claimed = s_n;
    const unsigned long long t_tile = threadIdx.x == 0 ? global_ns() : 0ull;
    // the pair state and pass data were released before this claim became possible; read them from L2
    const int phase = __ldcg(&a.pairs[p].phase);
    const PairState& tps = stage_state(a, p, smem + (phase == kPhaseEval ? kSmStateB : kSmStateA));
    const SlotInfo& sb = a.slots[2 * p];
    const SlotInfo& sa = a.slots[2 * p + 1];
    if (phase == kPhaseNeedNN) iter_tile<true>(a, tps, sb, sa, p, tile0, smem);            // one tile per claim
    else if (phase == kPhaseFitness) fitness_tile<true>(a, tps, sb, sa, p, tile0, smem);   // one tile per claim
    else
      for (uint32_t k = 0; k < n_claimed; ++k) {
        if (k) __syncthreads();  // the previous tile's partial sums have left the scratch
        eval_tile<true>(a, tps, sb, sa, p, tile0 + k, smem);
      }
    __syncthreads();
    if (threadIdx.x == 0) {  // release: these tiles' partial sums, correspondences, matrices and hints come before their tickets
      const uint32_t n_live = (sa.n_pts + kIterTile - 1) / kIterTile;
      s_last = atom_add_release(&a.pairs[p].ticket, n_claimed) + n_claimed == n_live;
      atomicAdd(&a.ctl[0], n_claimed);
      atomicAdd(&a.ctl[phase == kPhaseNeedNN ? 4 : (phase == kPhaseEval ? 5 : 6)], (uint32_t)(global_ns() - t_tile));  // statistics: ns in tiles by pass type
    }
    __syncthreads();
    if (s_last) {  // this CTA delivered the last tile of the pass: control step, then publish what comes next
      const unsigned long long t_ctrl = threadIdx.x == 0 ? global_ns() : 0ull;
      uint32_t next_tiles = 0;
      if (phase == kPhaseFitness) {
        fitness_finish(a, p, smem);
      } else {
        ctrl_step_body(a, p, phase == kPhaseEval, smem);
        next_tiles = (sa.n_pts + kIterTile - 1) / kIterTile;  // search, trial and fitness passes all cover the moving cloud
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        atomicAdd(&a.ctl[1], 1u);
        const int next_phase = next_tiles ? reinterpret_cast<const CtrlShared*>(smem)->ps.phase : kPhaseFinished;
        // several trial tiles per claim only when there are more tiles in flight than CTAs (a single pair has fewer: one tile per CTA)
        const bool crowded = (unsigned long long)a.n_pairs * next_tiles > 2ull * gridDim.x;
        publish_pass(a, p, next_tiles, next_phase == kPhaseEval && crowded ? kTrialTilesPerClaim : 1u);
        atomicAdd(&a.ctl[7], (uint32_t)(global_ns() - t_ctrl));  // statistics: ns in control steps (incl. publishing)
        if (next_tiles == 0) red_add_release(&a.flags[1], -1);  // the pair is closed: its results come before the count
      }
    }
    __syncthreads();
  }
}

// THROUGHPUT mode — the chunks of a batch call, several streams per device.  The same tile and control functions, but one
// kernel per pass and a separate (tiny) control kernel, replayed by the WHILE node of a CUDA graph until no pair iterates:
//     search -> control -> trial -> control -> trial -> control -> condition
// No host poll either, but nothing waits on the device: while one chunk sits in a control kernel (one CTA per pair) the SMs run
// the search kernels of the other chunks, and the trial and control kernels have a light footprint.  Measured on B200 (64
// pairs, 16 scenes, loop only): persistent kernel 11.2 ms on one stream but 13.7-16.3 ms on six (its resident CTAs hold the
// registers of every SM, so the chunks serialise and each drags its own tail); per-pass kernels 14.9 ms on one stream and
// 10.3 ms on six (profiles/r02_summary.md).  Results are bit-identical in both modes (same tile partials, same control step).
__global__ void __launch_bounds__(kIterTile, 4) gicp_search_kernel(const __grid_constant__ GicpArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  const uint32_t p = blockIdx.y;
  if (__ldcg(&a.pairs[p].phase) != kPhaseNeedNN) return;
  const SlotInfo& sa = a.slots[2 * p + 1];
  // the grid is sized from an estimate of the filtered size (Workspace::grid_frac): a CTA strides over the tiles beyond it
  for (uint32_t tile = blockIdx.x; tile * kIterTile < sa.n_pts; tile += gridDim.x) {
    if (tile != blockIdx.x) __syncthreads();  // the previous tile is done with the scratch the state is staged into
    iter_tile<true>(a, stage_state(a, p, smem + kSmStateA), a.slots[2 * p], sa, p, tile, smem);
  }
}

// (Tried: the control step fused into this kernel by the ticket scheme — one launch less per trial pass, but the inlined FP64
// chain raises the kernel from 56 to 80+ registers and the light trial tiles lose a resident CTA per SM: 3262-3283 against
// 3294-3300 registrations/s, profiles/r02_summary.md.)
#ifndef S3D_TRIAL_MINB
#define S3D_TRIAL_MINB 4
#endif
__global__ void __launch_bounds__(kIterTile, S3D_TRIAL_MINB) gicp_trial_kernel(const __grid_constant__ GicpArgs a) {
  constexpr size_t kScratch = size_t(kIterTile) * 64 + 16 * kEvalSums * 8;
  __shared__ __align__(16) unsigned char smem[kScratch + sizeof(PairState)];
  const uint32_t p = blockIdx.y;
  if (__ldcg(&a.pairs[p].phase) != kPhaseEval) return;
  const SlotInfo& sa = a.slots[2 * p + 1];
  if (blockIdx.x * kIterTile >= sa.n_pts) return;
  const PairState& ps = stage_state(a, p, smem + kScratch);
  for (uint32_t tile = blockIdx.x; tile * kIterTile < sa.n_pts; tile += gridDim.x) {
    if (tile != blockIdx.x) __syncthreads();  // the previous tile's partial sums have left the scratch
    eval_tile<true>(a, ps, a.slots[2 * p], sa, p, tile, smem);
  }
}

// one CTA per pair; the first control launch of a round serves pairs that just searched, the later ones pairs that were just evaluated
__global__ void __launch_bounds__(256) gicp_ctrl_kernel(const __grid_constant__ GicpArgs a, int after_eval) {
  __shared__ __align__(16) unsigned char smem[sizeof(CtrlShared)];
  const uint32_t p = blockIdx.x;
  if (__ldcg(&a.pairs[p].phase) != (after_eval ? kPhaseEval : kPhaseNeedNN)) return;
  ctrl_step_body(a, p, after_eval, smem);
  __syncthreads();
  if (threadIdx.x == 0) {
    atomicAdd(&a.ctl[0], (a.slots[2 * p + 1].n_pts + kIterTile - 1) / kIterTile);  // statistics: tiles of the pass just summed
    atomicAdd(&a.ctl[1], 1u);
    if (reinterpret_cast<const CtrlShared*>(smem)->ps.phase == kPhaseFitness) atomicSub(&a.flags[1], 1);  // the outer loop of this pair has ended
  }
}

__global__ void gicp_cond_kernel(const __grid_constant__ GicpArgs a, cudaGraphConditionalHandle cond) {
  const uint32_t rounds = ++a.ctl[3];
  const bool stuck = rounds >= a.max_launches;
  if (stuck) atomicOr(&a.flags[0], kErrWatchdog);
  cudaGraphSetConditional(cond, (a.flags[1] > 0 && !stuck) ? 1u : 0u);
}

__global__ void __launch_bounds__(kIterTile, 4) gicp_fitness_kernel(const __grid_constant__ GicpArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  const uint32_t p = blockIdx.y;
  if (__ldcg(&a.pairs[p].phase) != kPhaseFitness) return;
  const SlotInfo& sa = a.slots[2 * p + 1];
  for (uint32_t tile = blockIdx.x; tile * kIterTile < sa.n_pts; tile += gridDim.x) {
    if (tile != blockIdx.x) __syncthreads();
    fitness_tile<true>(a, stage_state(a, p, smem + kSmStateA), a.slots[2 * p], sa, p, tile, smem);
  }
}

__global__ void __launch_bounds__(kIterTile) gicp_fitness_finish_kernel(const __grid_constant__ GicpArgs a) {
  __shared__ __align__(16) unsigned char smem[size_t(kIterTile) * 16];
  if (__ldcg(&a.pairs[blockIdx.x].phase) != kPhaseFitness) return;
  fitness_finish(a, blockIdx.x, smem);
  if (threadIdx.x == 0) atomicAdd(&a.ctl[0], (a.slots[2 * blockIdx.x + 1].n_pts + kIterTile - 1) / kIterTile);
}

// ------------------------------------------------------------------------------------------------------------------
static void iso_inverse(const double T[16], double out[16]) {
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) out[c * 4 + r] = T[r * 4 + c];
  for (int r = 0; r < 3; ++r) { double s = 0; for (int c = 0; c < 3; ++c) s += out[c * 4 + r] * T[12 + c]; out[12 + r] = -s; }
  out[3] = out[7] = out[11] = 0; out[15] = 1;
}
static void m4d_mul(const double A[16], const double B[16], double C[16]) {
  for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) { double s = 0; for (int k = 0; k < 4; ++k) s += A[k * 4 + r] * B[c * 4 + k]; C[c * 4 + r] = s; }
}
// Eigen::AngleAxisd(R).angle() — via the quaternion, in [0, pi]   (align() :168)
static double rotation_angle(const double T[16]) {
  const double m00 = T[0], m11 = T[5], m22 = T[10], m01 = T[4], m02 = T[8], m10 = T[1], m12 = T[9], m20 = T[2], m21 = T[6];
  double w, x, y, z;
  const double tr = m00 + m11 + m22;
  if (tr > 0) {
    double t = sqrt(tr + 1.0); w = 0.5 * t; t = 0.5 / t;
    x = (m21 - m12) * t; y = (m02 - m20) * t; z = (m10 - m01) * t;
  } else {
    int i = 0;
    if (m11 > m00) i = 1;
    if (m22 > (i == 0 ? m00 : m11)) i = 2;
    const double M[3][3] = {{m00, m01, m02}, {m10, m11, m12}, {m20, m21, m22}};
    const int j = (i + 1) % 3, k = (i + 2) % 3;
    double t = sqrt(M[i][i] - M[j][j] - M[k][k] + 1.0);
    double q[3];
    q[i] = 0.5 * t; t = 0.5 / t;
    w = (M[k][j] - M[j][k]) * t; q[j] = (M[j][i] + M[i][j]) * t; q[k] = (M[k][i] + M[i][k]) * t;
    x = q[0]; y = q[1]; z = q[2];
  }
  return 2.0 * atan2(sqrt(x * x + y * y + z * z), fabs(w));
}

double rotation_angle_of(const double T[16]) { return rotation_angle(T); }  // shared with ndt.cu

void check_arena(Workspace& ws, const int32_t* h_flags) {
  if (h_flags[0] & kErrSortStall) throw CudaError{"radix sort: look-back spin limit reached (scheduler fault)"};
  if (h_flags[0] & kErrHashArena) throw ArenaOverflow{(size_t)h_flags[3] + (size_t)h_flags[3] / 8 + 64};
}

static int loop_grid(const Workspace& ws) {
  const int sms = ws.n_sms;
  static const int per_sm = [] { const char* e = getenv("S3D_LOOP_CTAS_PER_SM"); return e ? std::max(1, atoi(e)) : 2; }();  // A/B measurements
  return std::max(1, sms) * per_sm;  // 2 resident CTAs per SM (128 registers, 46 KB shared memory)
}

// Throughput mode: WHILE (a pair iterates) { search, control, trial, control, trial, control, condition } as a CUDA graph with a
// conditional node.  The kernels read everything from the GicpArgs block at a fixed device address; only the grid dimensions
// depend on the batch, so executable graphs are cached per workspace by (grid tiles, tiles per pair, pairs).
static cudaGraphExec_t loop_graph_for(Workspace& ws, const GicpArgs& args, uint32_t tiles_per_pair, uint32_t grid_tiles, uint32_t np) {
  // the graphs hold the argument block by value: when a buffer has moved (the batch grew), the cached graphs are stale
  uint64_t sig = 1469598103934665603ull;
  {
    GicpArgs key_args = args;
    key_args.tiles_per_pair = 0; key_args.n_pairs = 0;
    const unsigned char* b = reinterpret_cast<const unsigned char*>(&key_args);
    for (size_t i = 0; i < sizeof key_args; ++i) { sig ^= b[i]; sig *= 1099511628211ull; }
  }
  // ... and a service that sees many batch shapes must not collect executable graphs without bound
  if (sig != ws.loop_graph_sig || ws.loop_graphs.size() >= 64) {
    for (auto& g : ws.loop_graphs) cudaGraphExecDestroy(g.second);
    for (cudaGraph_t g : ws.loop_graph_defs) cudaGraphDestroy(g);
    ws.loop_graphs.clear(); ws.loop_graph_defs.clear();
    ws.loop_graph_sig = sig;
  }
  const uint64_t key = (uint64_t)grid_tiles << 44 | (uint64_t)tiles_per_pair << 20 | np;
  auto it = ws.loop_graphs.find(key);
  if (it != ws.loop_graphs.end()) return it->second;
  cudaGraph_t graph;
  S3D_CUDA(cudaGraphCreate(&graph, 0));
  cudaGraphConditionalHandle handle;
  S3D_CUDA(cudaGraphConditionalHandleCreate(&handle, graph, 1, cudaGraphCondAssignDefault));  // every replay starts with "true"
  cudaGraphNodeParams cp = {};
  cp.type = cudaGraphNodeTypeConditional;
  cp.conditional.handle = handle;
  cp.conditional.type = cudaGraphCondTypeWhile;
  cp.conditional.size = 1;
  cudaGraphNode_t cond_node;
  S3D_CUDA(cudaGraphAddNode(&cond_node, graph, nullptr, 0, &cp));
  cudaGraph_t body = cp.conditional.phGraph_out[0];
  GicpArgs ap = args;
  int zero = 0, one = 1;
  cudaGraphNode_t prev = nullptr;
  auto add = [&](void* fn, dim3 grid, unsigned block, unsigned smem, void** args) {
    cudaKernelNodeParams kp = {};
    kp.func = fn; kp.gridDim = grid; kp.blockDim = dim3(block); kp.sharedMemBytes = smem; kp.kernelParams = args;
    cudaGraphNode_t node;
    S3D_CUDA(cudaGraphAddKernelNode(&node, body, prev ? &prev : nullptr, prev ? 1 : 0, &kp));
    prev = node;
  };
  void* a1[] = {&ap};
  void* a_ctrl0[] = {&ap, &zero};
  void* a_ctrl1[] = {&ap, &one};
  void* a_cond[] = {&ap, &handle};
  const dim3 tiles(grid_tiles, np);
  add(reinterpret_cast<void*>(gicp_search_kernel), tiles, kIterTile, (unsigned)kSmTile, a1);
  add(reinterpret_cast<void*>(gicp_ctrl_kernel), dim3(np), 256, 0, a_ctrl0);
  for (int e = 0; e < 2; ++e) {  // two trial/advance passes per round: most outer iterations finish within one round
    add(reinterpret_cast<void*>(gicp_trial_kernel), tiles, kIterTile, 0, a1);
    add(reinterpret_cast<void*>(gicp_ctrl_kernel), dim3(np), 256, 0, a_ctrl1);
  }
  add(reinterpret_cast<void*>(gicp_cond_kernel), dim3(1), 1, 0, a_cond);
  cudaGraphExec_t exec;
  S3D_CUDA(cudaGraphInstantiate(&exec, graph, 0));
  ws.loop_graphs[key] = exec;
  ws.loop_graph_defs.push_back(graph);
  return exec;
}

// Runs the GICP loop + fitness for every pair of the batch (grids and covariances must be ready) and fills `out`
// with the decisions of doICP (:74-77) and align() (:134-135, :167-172).  Latency mode (single calls): set-up kernel + ONE
// persistent loop kernel.  Throughput mode (the chunks of a batch call, several streams per device): set-up kernel + one graph
// replay (per-pass kernels inside a WHILE node) + the fitness kernels.  With stage profiling on, the throughput kernels are
// launched from the host instead, round by round with one poll each, so that every kernel can be bracketed by events.
void run_gicp(Workspace& ws, const std::vector<s3d_registration_parameters>& params, const double* guesses, s3d_result* out) {
  const uint32_t np = ws.n_pairs;
  if (np == 0) return;
  cudaStream_t st = ws.stream;
  const uint32_t max_na = ws.max_na;
  const uint32_t tiles_per_pair = std::max<uint32_t>(1, (max_na + kIterTile - 1) / kIterTile);
  ws.pairs.reserve(sizeof(PairState) * np);
  ws.h_pairs.reserve(sizeof(PairState) * np);
  ws.moved.reserve(16 * std::max<size_t>(ws.total, 4));
  ws.prev_nn.reserve(4 * std::max<size_t>(ws.total, 4));
  ws.sec_lb.reserve(4 * std::max<size_t>(ws.total, 4));
  ws.moments.reserve(sizeof(double) * kNumMoments * size_t(tiles_per_pair) * np);
  ws.eval_part.reserve(sizeof(double) * kEvalSums * kLineSearchTrials * size_t(tiles_per_pair) * np);
  ws.corr.reserve(4 * std::max<size_t>(ws.total, 4));
  ws.mahal.reserve(48 * std::max<size_t>(ws.total, 4));
  ws.fit_partial.reserve(sizeof(double) * 2 * size_t(tiles_per_pair) * np);
  ws.gicp_sched.reserve(sizeof(PairSched) * np + 64);
  PairState* hp = ws.h_pairs.as<PairState>();
  for (uint32_t p = 0; p < np; ++p) {
    const s3d_registration_parameters& cfg = params[p];
    PairState& ps = hp[p];
    memset(&ps, 0, sizeof ps);
    for (int i = 0; i < 16; ++i) {
      ps.guess[i] = (float)guesses[16 * p + i];  // guess.matrix().cast<float>()  :70
      ps.T[i] = ps.prev[i] = ps.final_T[i] = (i % 5 == 0) ? 1.f : 0.f;
    }
    ps.max_corr2 = cfg.max_correspondence_distance * cfg.max_correspondence_distance;
    ps.rot_eps = cfg.rotation_epsilon; ps.trans_eps = cfg.transformation_epsilon;
    ps.fit_range = cfg.max_correspondence_distance;
    ps.pt_off = ws.pair_off[p];
    ps.max_iter = cfg.maximum_iterations; ps.max_inner = cfg.maximum_optimizer_iterations; ps.k = cfg.correspondence_randomness;
    ps.optimizer = ws.gicp_optimizer;
  }
  S3D_CUDA(cudaMemcpyAsync(ws.pairs.p, hp, sizeof(PairState) * np, cudaMemcpyHostToDevice, st));
  const SlotInfo* slots = ws.slots.as<SlotInfo>();
  PairState* pairs = ws.pairs.as<PairState>();
  int32_t* flags = ws.flags.as<int32_t>();
  int32_t* h_flags = ws.h_small.as<int32_t>();
  uint32_t* h_ctl = ws.h_small.as<uint32_t>() + 8;
  uint32_t* ctl = ws.gicp_sched.as<uint32_t>();                                       // 16 words of counters ...
  PairSched* psched = reinterpret_cast<PairSched*>(ws.gicp_sched.as<char>() + 64);    // ... then one scheduler entry per pair
  static const unsigned long long watchdog = [] {  // cycles without finding work after which the loop kernel gives up (~3 s; a loop takes milliseconds)
    const char* e = getenv("S3D_WATCHDOG_MCYCLES");
    return (e ? (unsigned long long)atoll(e) : 6000ull) * 1000000ull;
  }();
  // S3D_LOOP_MODE (measurement aid): 0 = by call type (default), 1 = always the persistent launch, 2 = always the per-pass kernels (graph replay),
  // 3 = the per-pass kernels launched from the host with one poll per round (what stage profiling uses)
  const char* loop_env = getenv("S3D_LOOP_MODE");
  const int loop_mode = loop_env ? atoi(loop_env) : 0;
  const uint32_t linger = 0;
  const bool throughput = loop_mode == 2 || loop_mode == 3 || (loop_mode == 0 && ws.blocking_sync);
  GicpArgs args_value;
  GicpArgs* ha = &args_value;
  *ha = GicpArgs{slots, pairs, ws.moved.as<float4>(), ws.prev_nn.as<uint32_t>(), ws.sec_lb.as<float>(), ws.corr.as<uint32_t>(), ws.mahal.as<double>(),
                 ws.moments.as<double>(), ws.eval_part.as<double>(), ws.fit_partial.as<double>(), flags, psched, ctl, tiles_per_pair, np,
                 linger, 1u << 20, watchdog};
  S3D_CUDA(cudaMemsetAsync(ctl, 0, 64, st));
  // launch grid: the tiles the filtered clouds are expected to have (the kernels stride over what a short grid leaves), in steps
  // of 16 tiles so that the cached graphs stay few
  const uint32_t grid_tiles = std::min<uint32_t>(tiles_per_pair, (ws.grid_x(tiles_per_pair, np, 4) + 15u) & ~15u);
  dim3 grid(std::max<uint32_t>(1, grid_tiles), np);
  {
    StageTimer timer(ws, kStageSolve);
    gicp_prepare_kernel<<<grid, 256, 0, st>>>(slots, pairs, ws.moved.as<float4>(), ws.prev_nn.as<uint32_t>(), ws.sec_lb.as<float>(), psched, flags);
    ++ws.launches;
  }
  const GicpArgs dargs = *ha;
  if (!throughput) {
    StageTimer timer(ws, kStageIter);
    gicp_loop_kernel<<<loop_grid(ws), kIterTile, kSmLoop, st>>>(dargs);
    ++ws.launches;
    S3D_CUDA(cudaGetLastError());
  } else {
    if (!ws.profiling && loop_mode != 3) {
      StageTimer timer(ws, kStageIter);
      S3D_CUDA(cudaGraphLaunch(loop_graph_for(ws, dargs, tiles_per_pair, grid_tiles, np), st));
    } else {
      // the same kernels from the host, one poll per round, so that each can be timed
      for (uint32_t round = 0; round < (1u << 20); ++round) {
        {
          StageTimer timer(ws, kStageIter);
          gicp_search_kernel<<<grid, kIterTile, kSmTile, st>>>(dargs);
          ++ws.launches;
        }
        {
          StageTimer timer(ws, kStageSolve);
          gicp_ctrl_kernel<<<np, 256, 0, st>>>(dargs, 0);
          for (int e = 0; e < 2; ++e) {
            gicp_trial_kernel<<<grid, kIterTile, 0, st>>>(dargs);
            gicp_ctrl_kernel<<<np, 256, 0, st>>>(dargs, 1);
          }
          ws.launches += 5;
        }
        S3D_CUDA(cudaMemcpyAsync(h_flags, flags, 16, cudaMemcpyDeviceToHost, st));
        ws.sync();
        ws.d2h += 16;
        if (h_flags[1] <= 0) break;
      }
    }
    {
      StageTimer timer(ws, kStageFitness);
      gicp_fitness_kernel<<<grid, kIterTile, kSmTile, st>>>(dargs);
      gicp_fitness_finish_kernel<<<np, kIterTile, 0, st>>>(dargs);
      ws.launches += 2;
    }
    S3D_CUDA(cudaGetLastError());
  }
  S3D_CUDA(cudaMemcpyAsync(h_ctl, ctl, 32, cudaMemcpyDeviceToHost, st));
  S3D_CUDA(cudaMemcpyAsync(hp, pairs, sizeof(PairState) * np, cudaMemcpyDeviceToHost, st));
  SlotInfo* hs = ws.h_slots.as<SlotInfo>();
  S3D_CUDA(cudaMemcpyAsync(hs, slots, sizeof(SlotInfo) * ws.n_slots, cudaMemcpyDeviceToHost, st));
  S3D_CUDA(cudaMemcpyAsync(h_flags, flags, 16, cudaMemcpyDeviceToHost, st));
  ws.sync();
  ws.d2h += sizeof(PairState) * np + sizeof(SlotInfo) * ws.n_slots + 32;
  ws.passes += h_ctl[0]; ws.ctrl_steps += h_ctl[1];
  if (ws.n_tiles > 0) ws.learn_grid_frac(hs, ws.n_slots);  // raw-cloud batch: how much of the raw clouds survived the voxel filter sizes the next batch's grids
  if (getenv("S3D_LOOP_STATS") && !throughput)
    fprintf(stderr, "[s3d loop] pairs %u tiles %u control steps %u | per control step %.1f us | CTA-time in search tiles %.0f us, trial tiles %.0f us, fitness tiles %.0f us\n",
            np, h_ctl[0], h_ctl[1], h_ctl[1] ? 1e-3 * h_ctl[7] / h_ctl[1] : 0.0, 1e-3 * h_ctl[4], 1e-3 * h_ctl[5], 1e-3 * h_ctl[6]);
  ws.launches += 7ull * h_ctl[3];  // rounds replayed by the graph's WHILE node (throughput mode): 7 kernels each
  for (auto& sp : ws.spans) if (sp.stage == kStageIter && h_ctl[3]) sp.n_launch = 7 * h_ctl[3];
  ws.collect_spans();
  check_arena(ws, h_flags);
  if (h_flags[0] & kErrWatchdog) throw CudaError{"GICP loop kernel: watchdog expired (scheduler fault)"};
  for (uint32_t p = 0; p < np; ++p) {
    const s3d_registration_parameters& cfg = params[p];
    const PairState& ps = hp[p];
    s3d_result& r = out[p];
    memset(&r, 0, sizeof r);
    for (int i = 0; i < 16; ++i) r.T[i] = (i % 5 == 0) ? 1.0 : 0.0;
    r.n_source = hs[2 * p].n_pts; r.n_target = hs[2 * p + 1].n_pts;
    if (r.n_target < 100 || r.n_source < 100) { r.status = S3D_TOO_FEW_POINTS; continue; }  // :134-135
    if (ps.active) {  // the loop kernel left the pair unfinished: a scheduler / optimiser fault, not a NoMatch
      r.status = S3D_INTERNAL_ERROR;
      set_error("GICP loop ended with an active pair");
      continue;
    }
    for (int i = 0; i < 16; ++i) r.T[i] = (double)ps.final_T[i];  // Transform(Eigen::Isometry3f(final))  :80
    r.fitness = ps.fit_n > 0 ? ps.fit_sum / (double)ps.fit_n : 1.7976931348623157e308;
    r.converged = ps.converged; r.outer_iterations = ps.outer_iterations; r.inner_iterations = ps.inner_iterations;
    r.n_correspondences = ps.n_corr;
    if (!ps.converged || r.fitness > cfg.max_fitness_score) { r.status = S3D_NOT_CONVERGED; continue; }  // :74-77
    double ginv[16], delta[16];
    iso_inverse(guesses + 16 * p, ginv);
    m4d_mul(ginv, r.T, delta);
    const double tn = sqrt(delta[12] * delta[12] + delta[13] * delta[13] + delta[14] * delta[14]);
    r.status = (tn > cfg.max_translation || rotation_angle(delta) > cfg.max_rotation) ? S3D_TOO_FAR_FROM_GUESS : S3D_OK;  // :167-172
  }
}

}  // namespace s3d
