// internal.h — host-side plumbing shared by the .cu files of libs3d_b200.so (not part of the public C-ABI).
#pragma once

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/s3d_b200.h"
#include "common.cuh"
#include "gicp_math.h"

namespace s3d {

void set_error(const std::string& msg);  // thread-local message behind s3d_last_error()

struct CudaError { std::string what; };
struct ArenaOverflow { size_t needed; };  // the hash arena was too small for this batch; re-run with `needed` entries
#define S3D_CUDA(expr)                                                                                         \
  do {                                                                                                         \
    cudaError_t _e = (expr);                                                                                   \
    if (_e != cudaSuccess) throw ::s3d::CudaError{std::string(#expr) + ": " + cudaGetErrorString(_e)};         \
  } while (0)

// growable device buffer (grow-only; reused across calls so steady state does no cudaMalloc)
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  void reserve(size_t bytes) {
    if (bytes <= cap) return;
    if (p) S3D_CUDA(cudaFree(p));
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    S3D_CUDA(cudaMalloc(&p, want));
    cap = want;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <typename T> T* as() const { return static_cast<T*>(p); }
};

struct PinnedBuf {
  void* p = nullptr;
  size_t cap = 0;
  void reserve(size_t bytes) {
    if (bytes <= cap) return;
    if (p) S3D_CUDA(cudaFreeHost(p));
    p = nullptr; cap = 0;
    S3D_CUDA(cudaMallocHost(&p, bytes + bytes / 4 + 256));
    cap = bytes + bytes / 4 + 256;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
  template <typename T> T* as() const { return static_cast<T*>(p); }
};

// Device-resident state of one registration (pair of slots).
struct PairState {
  float  guess[16];        // guess.matrix().cast<float>()   PointCloudSensor.cpp:70
  float  T[16];            // transformation_
  float  prev[16];         // previous_transformation_
  float  final_T[16];      // final_transformation_ = previous * guess
  float  T_search[16];     // the transformation_ the last correspondence search ran with (temporal-coherence certificate)
  double RRt[3][3];        // (T*guess).R (T*guess).R^T for the Mahalanobis matrices of this iteration
  double R[3][3];
  double max_corr2;        // corr_dist_threshold_^2
  double rot_eps, trans_eps;
  double fit_range;        // getFitnessScore(max_range): squared distance compared with this un-squared value
  double fit_sum;
  uint32_t fit_n;
  int32_t max_iter, max_inner, k;
  int32_t optimizer;       // S3D_GICP_NEWTON / S3D_GICP_BFGS: which inner optimiser runs (the context's setting)
  union {                  // resumable inner optimiser: one at a time, so they share storage
    NewtonState nst;       // PCL >= 1.14 estimateRigidTransformationNewton (gicp_math.h)
    BfgsState bst;         // PCL <= 1.13 estimateRigidTransformationBFGS (gicp_bfgs.h)
  };
  float  T_eval[16];       // float matrix of the outer iteration's start state x0 (PCL applyState), evaluated by the search pass
  float  T_trial[kLineSearchTrials][16];  // float matrices of the back-tracking trials x - 2^-j delta of the current Newton step
                                          // (BFGS: T_trial[0] is the one pending line-search trial x0 + alpha p)
  int32_t trial_first, trial_count;       // trials the next evaluation pass has to cover (0,1 first; 1,9 if trial 0 failed; BFGS: 0,1)
  double sums[kNumMoments];// reduced sums of the current correspondence set (static part) + last evaluation (residual part)
  int32_t phase;           // kPhaseNeedNN / kPhaseEval / kPhaseFitness / kPhaseFinished
  int32_t active;          // 1 while the outer loop runs
  int32_t converged;
  int32_t failed;          // optimiser exception (<4 correspondences)
  int32_t outer_iterations, inner_iterations;
  uint32_t n_corr;
  uint32_t pt_off;         // first index of this pair in the per-pair arrays (moved, prev_nn, sec_lb, corr, mahal)
  uint32_t ticket;         // tiles of the running pass that have delivered their partial sums (the last one runs the control step)
};
static_assert(sizeof(PairState) % 8 == 0, "PairState is staged through shared memory in 8-byte words");

// Scheduler entry of one pair in the persistent GICP loop kernel (gicp.cu): both words are epoch << 32 | count.
struct PairSched {
  unsigned long long claim;  // next unclaimed tile of the open pass
  unsigned long long desc;   // tiles of the open pass (0: nothing to claim)
};

// Arguments of the GICP loop kernels, passed BY VALUE as a kernel parameter: pointers that arrive in parameter space are known to
// be global (LDG / STG); the same pointers read from a block in device memory compile to generic LD / ST (measured: the search
// kernel 5 % slower).  The cached loop graphs therefore hold these values, and are dropped when a workspace buffer moves.
struct GicpArgs {
  const SlotInfo* __restrict__ slots; PairState* __restrict__ pairs;
  const float4* __restrict__ moved; uint32_t* __restrict__ prev_nn; float* __restrict__ sec_lb; uint32_t* __restrict__ corr; double* __restrict__ mahal;
  double* __restrict__ moments; double* __restrict__ eval_part; double* __restrict__ fit_partial;
  int32_t* __restrict__ flags;          // [0] error bits, [1] active pairs
  PairSched* __restrict__ psched;
  uint32_t* __restrict__ ctl;           // [0] tiles processed, [1] control steps (statistics); [3] rounds (throughput mode)
  uint32_t tiles_per_pair, n_pairs;
  uint32_t reserved;
  uint32_t max_launches;   // throughput mode: rounds after which the loop gives up (scheduler fault)
  unsigned long long watchdog_cycles;
};

constexpr int kIterTile = 256;   // source points per CTA in the fused correspondence kernel

struct NdtLeaf;  // ndt_math.h

// NDT target grid of one fixed cloud: pcl::VoxelGridCovariance at `resolution` (ndt.cu).  Built in a workspace for the fixed
// clouds of a raw NDT batch, or for every cloud of s3d_prepare_clouds_ndt, whose handles keep it beside their copies of the leaves
// and the hash table.  Hash entries are (voxel key, leaf rank) with ranks relative to `leaves`, so a copy of both arrays is valid.
struct NdtGrid {
  float resolution, inv_leaf;
  int32_t min_b[3], div_b[3];
  uint32_t mul1, mul2;
  uint32_t n_voxels;         // occupied voxels = entries of `leaves`
  uint32_t n_leaves;         // voxels with >= 6 points: the centroid cloud
  uint32_t hash_mask;        // entries of `table` - 1
  uint32_t escaped;          // some float centroid lies outside its own voxel
  int32_t searchable;        // grid parameters valid (finite cloud, no int32 overflow)
  uint32_t reserved;
  NdtLeaf* leaves;           // n_voxels leaves in ascending key order
  uint2* table;              // open-addressing hash voxel key -> leaf rank
};

// Which slots of a workspace batch get an NDT grid, and where it goes: slot s has one iff (s & skip_mask) == 0, grid s >> shift.
// Raw NDT batches build the grid of every fixed cloud (slot 2p -> grid p); the prepare pass builds one per slot.
struct NdtGridMap {
  uint32_t shift, skip_mask;
  __host__ __device__ bool has(uint32_t slot) const { return (slot & skip_mask) == 0; }
  __host__ __device__ uint32_t grid(uint32_t slot) const { return slot >> shift; }
  __host__ __device__ uint32_t slot(uint32_t g) const { return g << shift; }
};
constexpr NdtGridMap kNdtFixedSlots{1, 1}, kNdtEverySlot{0, 0};

// All device memory of one in-flight batch on one device.
struct Workspace {
  int device = 0;
  int n_sms = 148;                            // cudaDevAttrMultiProcessorCount of `device` (grid sizes of the grid-stride kernels)
  cudaStream_t stream = nullptr;
  cudaEvent_t sync_event = nullptr;           // cudaEventBlockingSync: a worker of a batch call sleeps in sync() instead of spinning on the stream
  bool blocking_sync = false;                 // set for the chunks of multi-threaded batch calls (many host threads per device, several ranks per box)
  cudaEvent_t input_event = nullptr;          // orders this workspace's stream after the caller's stream (s3d_set_input_stream)
  cudaStream_t input_stream = nullptr; bool wait_input = false;
  std::mutex* upload_gate = nullptr;          // when set, setup_batch holds it from its first host-to-device copy until the copies have landed
  // sizes of the current batch
  uint32_t n_slots = 0, n_pairs = 0, total = 0, n_tiles = 0;
  std::vector<uint32_t> h_off, h_n;           // per slot
  std::vector<uint32_t> pair_off;             // per pair: offset into the per-pair arrays
  uint32_t max_na = 0;                        // largest moving cloud of the batch (upper bound of the iteration grid)
  DevBuf slots, pairs;                        // SlotInfo[n_slots], PairState[n_pairs]
  DevBuf raw_stage;                           // float4[total]   H2D landing zone for host inputs
  DevBuf work, gpts;                          // float4[total]
  DevBuf keys0, keys1, vals0, vals1;          // uint32[total]
  DevBuf hist;                                // uint64[n_tiles*256]: look-back status words of the radix sort (sort.cuh), zero when (re)allocated
  DevBuf sort_totals;                         // uint32[4 passes * n_slots * 256] digit totals + 4 tile tickets
  // Launch grids are sized on the host from RAW cloud sizes, but the kernels behind the voxel filter work on the filtered clouds
  // (36 % of the points for a 0.1 m leaf on a 64-beam scan): two thirds of the CTAs of every kNN / search / trial / fitness launch
  // found nothing to do.  Those kernels now stride over their tiles, so ANY grid is correct, and the grid is sized with the
  // filtered / raw ratio the previous batch on this workspace showed (1 until one has run; S3D_GRID_FRAC pins it for A/B runs).
  // The ratio depends on the leaf size, so it is remembered per leaf (a loop-closure call alternates 0.5 m and 0.1 m passes).
  std::map<float, float> learned_frac;        // leaf size -> what the last raw-cloud batch with that leaf showed (+ margin)
  float batch_leaf = 0.f;                     // leaf size of the current batch (set by run_voxel)
  float grid_frac = 1.f;                      // what the current batch uses (1 for prepared clouds: their sizes are exact)
  int gicp_optimizer = S3D_GICP_NEWTON;       // inner optimiser of the GICP loop: the context's setting at the time the workspace was leased
  int ndt_omp_search = S3D_NDT_OMP_KDTREE;    // neighbour search of NDT_OMP: the context's setting at the time the workspace was leased
  // after a batch: `hs` = the slot table read back from the device
  void learn_grid_frac(const SlotInfo* hs, uint32_t ns) {
    if (!(batch_leaf > 0.f)) return;
    float frac = 0.f;
    for (uint32_t s = 0; s < ns; ++s)
      if (hs[s].n_raw > 0) frac = std::max(frac, (float)hs[s].n_pts / (float)hs[s].n_raw);
    if (frac > 0.f) learned_frac[batch_leaf] = std::min(1.f, frac * 1.08f + 1.f / 64.f);
  }
  // grid.x for a launch of `units` work items per cloud / pair over `rows` clouds / pairs: the estimate, but never so small that the
  // launch could not fill the GPU (`per_sm` CTAs per SM) when the bound allows it
  uint32_t grid_x(uint32_t units, uint32_t rows, uint32_t per_sm) const {
    const uint32_t est = (uint32_t)ceilf(units * grid_frac);
    const uint32_t fill = (uint32_t)((size_t(n_sms) * per_sm + rows - 1) / (rows ? rows : 1));
    return std::max<uint32_t>(1, std::min<uint32_t>(units, std::max(est, fill)));
  }
  uint32_t sort_epoch = 0;                    // bumped once per sort pass: tags the status words, so that they are never cleared
  size_t status_words = 0;
  DevBuf long_runs;                           // uint4[total/64]  voxels with more than 64 points: (slot, first sorted position, output rank)
  DevBuf tile_slot, tile_first, slot_tile_begin, tile_heads;
  DevBuf hash;                                // HashEntry[hash_cap]
  size_t hash_cap = 0;
  size_t hash_want = 0;                       // entries requested by the last arena overflow (0: default sizing)
  DevBuf knn_arena;                           // uint64[k * threads of the launch]: kNN heaps in global memory when k > kMaxKShared
  DevBuf normals;                             // double[total*4]  unit normal of the regularised covariance (+pad)
  DevBuf moved;                               // float4[total]   guess * A (Morton order of A)
  DevBuf prev_nn;                             // uint32[total]   last correspondence (warm start bound)
  DevBuf sec_lb;                              // float[total]    lower bound of the distance to every OTHER fixed point at the last search position
  DevBuf moments;                             // double[iter_tiles * 74]
  DevBuf eval_part;                           // double[iter_tiles * 13]
  DevBuf corr;                                // uint32[total]   correspondence of the current outer iteration (kNoIndex: none)
  DevBuf mahal;                               // double[total*6] Mahalanobis matrix of each correspondence
  DevBuf iter_tile_pair, iter_tile_first;     // uint32[iter_tiles]
  uint32_t iter_tiles = 0;
  DevBuf fit_partial;                         // double[iter_tiles*2]
  DevBuf accu, accu2, map_aux;                // map building: accumulated cloud, filtered cloud, poses / keep flags
  DevBuf ndt_pairs, ndt_leaves, ndt_hash, ndt_part;  // NDT: NdtPair[n_pairs], NdtLeaf[], uint2 hash arena, double[tiles * 44]
  DevBuf ndt_grids;                           // NdtGrid[]: the grids a build writes, or the grids of the pairs of an NDT align
  DevBuf ransac, ransac_idx;                  // RANSAC plane fit (ransac.cu): sampler state + one block of planes / flags / counts; uint32[n] shuffled indices
  DevBuf gicp_args, gicp_sched;               // GicpArgs; 16 counter words + PairSched[n_pairs] of the loop kernel
  uint64_t passes = 0, ctrl_steps = 0;        // tiles processed / control steps run by the loop kernel (statistics)
  std::map<uint64_t, cudaGraphExec_t> loop_graphs;  // throughput mode: WHILE (a pair iterates) { per-pass kernels }, by (tiles per pair, pairs)
  std::vector<cudaGraph_t> loop_graph_defs;
  uint64_t loop_graph_sig = 0;                // hash of the pointer values the cached graphs were built with
  DevBuf flags;                               // int32[16]: [0] error bits, [1] active pairs, [2] hash entries used, [3] entries needed, [8] long voxel runs, [9] kept points
  PinnedBuf h_slots, h_pairs, h_small, h_tiles, h_grids;  // pinned host mirrors
  PinnedBuf h_bounce;                            // pinned landing zone for pageable host clouds (setup_batch)
  PinnedBuf h_ransac;                            // one block of RANSAC planes / flags / counts read back for the replay
  uint64_t launches = 0, h2d = 0, d2h = 0;
  // optional stage timing (s3d_set_profiling)
  bool profiling = false;
  struct Span { int stage; cudaEvent_t a, b; uint32_t n_launch; };
  std::vector<Span> spans;
  std::vector<cudaEvent_t> event_pool;
  double stage_ms[S3D_N_STAGES] = {0, 0, 0, 0, 0, 0};
  uint64_t stage_launches[S3D_N_STAGES] = {0, 0, 0, 0, 0, 0};
  cudaEvent_t get_event();
  void collect_spans();  // after a stream synchronise

  void init(int dev);
  void destroy();
  SortState sort_state() { return SortState{sort_totals.as<uint32_t>(), hist.as<uint64_t>(), status_words, &sort_epoch, flags.as<int32_t>()}; }
  void sync();  // wait for everything enqueued on `stream`
  void order_after_input();  // s3d_set_input_stream: enqueue a wait for what the caller's stream holds now
};

enum ErrorBits { kErrHashArena = 1, kErrWatchdog = 2, kErrSortStall = 4 };
enum PairPhase { kPhaseNeedNN = 0, kPhaseEval = 1, kPhaseFinished = 2, kPhaseFitness = 3 };
constexpr int kEvalSums = 13;  // sums 60..72 of gicp_math.h: the residual-dependent part of an evaluation (per trial)
enum Stage { kStageVoxel = 0, kStageGrid = 1, kStageKnn = 2, kStageIter = 3, kStageSolve = 4, kStageFitness = 5 };

// RAII: brackets the kernels launched in its scope with two events when profiling is on
struct StageTimer {
  Workspace& ws; int stage; uint64_t l0; cudaEvent_t a = nullptr;
  StageTimer(Workspace& w, int s) : ws(w), stage(s), l0(w.launches) {
    if (ws.profiling) { a = ws.get_event(); cudaEventRecord(a, ws.stream); }
  }
  ~StageTimer() {
    if (a) { cudaEvent_t b = ws.get_event(); cudaEventRecord(b, ws.stream); ws.spans.push_back({stage, a, b, (uint32_t)(ws.launches - l0)}); }
  }
};

// ---- stage launchers (each enqueues kernels on ws.stream; no host synchronisation inside) -----------------
void setup_batch(Workspace& ws, const std::vector<const float*>& clouds, const std::vector<uint64_t>& sizes, uint32_t n_pairs);
// voxel.cu: clouds[i] (host or device memory of any GPU, sizes[i] points) copied verbatim to dst[i] on ws.device; synchronises ws
void upload_clouds(Workspace& ws, const std::vector<const float*>& clouds, const std::vector<uint64_t>& sizes, const std::vector<float4*>& dst);
void run_voxel(Workspace& ws, float leaf, uint32_t* leaf_keys = nullptr);  // leaf <= 0: working cloud = raw cloud; leaf_keys: unsorted voxel keys (device, total)
void run_grid(Workspace& ws, float leaf_hint);      // NN grid on the working clouds
void run_knn_covariances(Workspace& ws, int k, uint32_t* knn_index, float* knn_dist2);  // outputs optional (device, slot-concatenated)
void run_expand_cov(Workspace& ws, double* cov_out);  // full 3x3 covariances per original index (stage API)
void run_nn_stage(Workspace& ws, uint32_t ref_slot, uint32_t qry_slot, const float* T16_dev, uint32_t* nn_index, float* nn_dist2);
uint32_t run_accumulate(Workspace& ws, const std::vector<const float*>& clouds, const std::vector<uint64_t>& sizes, const double* poses,
                        const double* second = nullptr);  // -> ws.accu; second: one more 4x4 applied to every (float-rounded) point
// map.cu: every patch of s3d_prepare_combined_measurements (arguments as there, validated) into ws.accu; patch p is
// [patch_off[p], patch_off[p + 1]).  patch_inv: n_patches x 16 doubles of patch_pose.inverse(), or NULL.  Synchronises ws.
const float4* run_patch_gather(Workspace& ws, const s3d_cloud* scans, const int32_t* member_scan, const double* member_poses,
                               const int32_t* patch_first_member, const double* patch_inv, uint32_t n_patches, std::vector<uint64_t>& patch_off);
uint32_t run_radius_filter(Workspace& ws, const float4* dev_in, uint32_t n, double radius, unsigned min_pts, float4* dev_out);
// map.cu: exclusive scan of n_tiles per-tile counts in place (one warp); *total = their sum
__global__ void keep_scan_kernel(uint32_t n_tiles, uint32_t* __restrict__ tile_counts, uint32_t* __restrict__ total);
// ransac.cu.  run_ransac_plane: RandomSampleConsensus + SampleConsensusModelPlane on the n device points (ransac_math.h); with
// want_inliers the ascending inlier indices are left at inliers_dev (workspace memory, valid until the next call on ws).
// run_ground_fill: the fill points of fillGroundPlane for the plane `coeff` and the loop values of ground_fill_lists().
struct RansacFit {
  bool ok = false;
  float coeff[4] = {0, 0, 0, 0};
  int32_t iterations = 0;
  uint64_t n_inliers = 0;
  uint32_t* inliers_dev = nullptr;
};
RansacFit run_ransac_plane(Workspace& ws, const float4* pts, uint32_t n, double threshold, int max_iterations, double probability,
                           bool want_inliers);
void run_ground_fill(Workspace& ws, const float coeff[4], const std::vector<double>& rings, const std::vector<double>& sin_a,
                     const std::vector<double>& cos_a, float4* dev_out);
void check_arena(Workspace& ws, const int32_t* h_flags);  // throws ArenaOverflow when the grid build flagged it (h_flags: synchronised copy)
void run_gicp(Workspace& ws, const std::vector<s3d_registration_parameters>& params, const double* guesses, s3d_result* out);
// ndt.cu.  run_ndt: doNDT for every pair of a raw batch (builds the grids of slots 2p).  run_ndt_grids: only the grids of the slots
// `map` selects, at `resolution`, into ws.ndt_grids (read back by the caller's next synchronise).  run_ndt_prepared: doNDT for
// pairs whose fixed-cloud grids exist: grids[p] is the grid of pair p (host records whose arrays live on the device).  direct7: the
// neighbourhood of pclomp's DIRECT7 search (NDT_OMP with S3D_NDT_OMP_DIRECT7) instead of PCL's radius search.
void run_ndt(Workspace& ws, const std::vector<s3d_registration_parameters>& params, const double* guesses, bool direct7, s3d_result* out);
void run_ndt_grids(Workspace& ws, NdtGridMap map, uint32_t n_grids, const float* resolution);
void run_ndt_prepared(Workspace& ws, const std::vector<s3d_registration_parameters>& params, const double* guesses, const NdtGrid* grids,
                      bool direct7, s3d_result* out);

}  // namespace s3d
