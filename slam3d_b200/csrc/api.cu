// api.cu — the C-ABI of include/s3d_b200.h: context, per-thread workspaces, batch sharding over devices.
//
// Mirrors the two arithmetic call sites of the reference (SURVEY 8b):
//   s3d_voxel_downsample  <-  PointCloudSensor::downsample            PointCloudSensor.cpp:190-201
//   s3d_gicp_align        <-  align() incl. doICP<GICP> and its gates  PointCloudSensor.cpp:52-82, 119-174
// Re-entrancy (ScanSensor.cpp:209-210 calls createConstraint from two threads): every call checks a private Workspace
// (device buffers + stream) out of the context's pool; there is no global mutable state.
// There is NO CPU fallback: without a CUDA device every entry point returns S3D_INTERNAL_ERROR.
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <thread>

#include "internal.h"
#include "ndt_math.h"
#include "ransac_math.h"

namespace s3d {

thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }

struct DeviceCtx {
  int device = 0;
  std::mutex mu;
  std::mutex upload_mu;  // one chunk uploads at a time (Workspace::upload_gate)
  std::vector<std::pair<void*, size_t>> free_blocks;  // recycled allocations of released prepared clouds
  uint64_t blocks_allocated = 0, blocks_reused = 0;   // prepared-cloud blocks from cudaMalloc / from free_blocks (under mu)
  std::vector<std::unique_ptr<Workspace>> pool;  // idle workspaces
  std::vector<Workspace*> all;
};

}  // namespace s3d

namespace s3d {
// Long-lived host threads of a context: batch calls hand their per-stream workers to the pool instead of spawning and
// joining std::threads on every call (round 1: 6 spawns per call and device).  A second batch call that arrives while the
// pool is busy (the API is re-entrant) falls back to threads of its own.
class WorkerPool {
 public:
  ~WorkerPool() {
    { std::lock_guard<std::mutex> g(mu_); stop_ = true; }
    cv_job_.notify_all();
    for (auto& t : threads_) t.join();
  }
  std::mutex call_mu;  // held by the batch call that owns the pool
  // runs f(0) .. f(n-1) concurrently, one index per thread, and returns when all have finished
  void run(int n, const std::function<void(int)>& f) {
    std::unique_lock<std::mutex> lk(mu_);
    while ((int)threads_.size() < n) { const int id = (int)threads_.size(); threads_.emplace_back([this, id] { loop(id); }); }
    job_ = &f; n_job_ = n; pending_ = n; ++generation_;
    cv_job_.notify_all();
    cv_done_.wait(lk, [this] { return pending_ == 0; });
    job_ = nullptr;
  }
 private:
  void loop(int id) {
    uint64_t seen = 0;
    std::unique_lock<std::mutex> lk(mu_);
    for (;;) {
      cv_job_.wait(lk, [&] { return stop_ || (generation_ != seen && id < n_job_); });
      if (stop_) return;
      seen = generation_;
      const std::function<void(int)>* f = job_;
      lk.unlock();
      (*f)(id);
      lk.lock();
      if (--pending_ == 0) cv_done_.notify_all();
    }
  }
  std::vector<std::thread> threads_;
  std::mutex mu_;
  std::condition_variable cv_job_, cv_done_;
  const std::function<void(int)>* job_ = nullptr;
  int n_job_ = 0, pending_ = 0;
  uint64_t generation_ = 0;
  bool stop_ = false;
};
}  // namespace s3d

struct s3d_prepared_cloud {
  int device_slot = 0;
  s3d::SlotInfo info;        // host copy; gpts / normals / table point into `block`
  void* block = nullptr;     // one device allocation: GICP [gpts | normals | hash table], NDT [gpts | hash table | NDT leaves | NDT hash]
  size_t block_bytes = 0;
  double density = 0;
  int k = 0;                 // kNN of the covariances (GICP handles); 0 for NDT handles
  float resolution = 0.f;    // NDT handles: resolution of `grid`; 0 for GICP handles
  s3d::NdtGrid grid{};       // NDT handles: the VoxelGridCovariance; leaves / table point into `block`
};

struct s3d_context {
  std::vector<std::unique_ptr<s3d::DeviceCtx>> devs;
  std::mutex mu;
  uint64_t launches = 0, h2d = 0, d2h = 0;
  uint64_t loop_tiles = 0, loop_ctrl_steps = 0;
  bool profiling = false;
  double stage_ms[S3D_N_STAGES] = {0, 0, 0, 0, 0, 0};
  uint64_t stage_launches[S3D_N_STAGES] = {0, 0, 0, 0, 0, 0};
  int max_pairs_per_launch = 32;
  // Host threads / streams per device.  Round 1 (host-driven rounds, one poll each) was fastest with 6; with the loop replayed by a
  // graph there is no host latency left to hide and 3-4 chunks are best (B200, 64 pairs: 3300 / 3294 / 3008 registrations/s with
  // 3 / 4 / 6 streams, e2e 2820 / 2831 / 2746; profiles/r02_summary.md).  The prepare + prepared-align path and the NDT branch
  // (252-register kernels) use 3.
  int streams_per_device = 4;
  int streams_small = 3;
  cudaStream_t input_stream = nullptr;  // s3d_set_input_stream: device-pointer inputs are produced on this stream
  bool have_input_stream = false;
  std::atomic<int> gicp_optimizer{S3D_GICP_NEWTON};  // s3d_set_gicp_optimizer
  std::atomic<int> ndt_omp_search{S3D_NDT_OMP_KDTREE};  // s3d_set_ndt_omp_search
  s3d::WorkerPool pool;
  // n workers through the pool, or through threads of the call's own when another batch call holds the pool
  void parallel(int n, const std::function<void(int)>& f) {
    std::unique_lock<std::mutex> lk(pool.call_mu, std::try_to_lock);
    if (lk.owns_lock()) { pool.run(n, f); return; }
    std::vector<std::thread> th;
    for (int i = 0; i < n; ++i) th.emplace_back([&f, i] { f(i); });
    for (auto& t : th) t.join();
  }
};

namespace s3d {

// Set by the worker threads of a batch call: their chunks take turns on the host-to-device link, so the first chunk is on the
// device after 1/W of the upload time and its kernels run while the next chunk uploads.  (Left to themselves the W streams
// share the link and all uploads end together, with the GPU idle until then: 64 pairs, 268 MB, measured in DESIGN.md 5.)
static thread_local bool t_gate_uploads = false;
static thread_local bool t_blocking_sync = false;  // worker of a multi-threaded batch call: sleep in Workspace::sync()

// Chunk size for `n` work items on W streams: the number of chunks is a multiple of W (every stream gets the same number of
// chunks — 4 chunks on 3 streams measured 15 % slower than 3 or 6) and no chunk exceeds `cap` items.
static int balanced_chunk(int n, int W, int cap) {
  if (n <= 0) return 1;
  const int waves = (n + W * cap - 1) / (W * cap);
  const int chunks = W * std::max(1, waves);
  return std::max(1, (n + chunks - 1) / chunks);
}

struct WsLease {
  s3d_context* ctx; DeviceCtx* dc; std::unique_ptr<Workspace> ws;
  WsLease(s3d_context* c, int slot) : ctx(c), dc(c->devs[slot].get()) {
    S3D_CUDA(cudaSetDevice(dc->device));
    {
      std::lock_guard<std::mutex> g(dc->mu);
      if (!dc->pool.empty()) { ws = std::move(dc->pool.back()); dc->pool.pop_back(); }
    }
    if (!ws) { ws.reset(new Workspace()); ws->init(dc->device); std::lock_guard<std::mutex> g(dc->mu); dc->all.push_back(ws.get()); }
    ws->profiling = ctx->profiling;
    ws->gicp_optimizer = ctx->gicp_optimizer.load();
    ws->ndt_omp_search = ctx->ndt_omp_search.load();
    static const bool gate_enabled = [] { const char* e = getenv("S3D_GATE_UPLOADS"); return !e || atoi(e) != 0; }();  // 0: A/B measurements
    ws->upload_gate = (t_gate_uploads && gate_enabled) ? &dc->upload_mu : nullptr;
    static const bool blocking_enabled = [] { const char* e = getenv("S3D_BLOCKING_SYNC"); return !e || atoi(e) != 0; }();  // 0: A/B measurements
    ws->blocking_sync = t_blocking_sync && blocking_enabled;
    ws->wait_input = ctx->have_input_stream; ws->input_stream = ctx->input_stream;
  }
  ~WsLease() {
    {
      std::lock_guard<std::mutex> g(ctx->mu);
      ctx->launches += ws->launches; ctx->h2d += ws->h2d; ctx->d2h += ws->d2h;
      ctx->loop_tiles += ws->passes; ctx->loop_ctrl_steps += ws->ctrl_steps;
      ws->launches = ws->h2d = ws->d2h = 0; ws->passes = ws->ctrl_steps = 0;
      if (ws->profiling) { cudaStreamSynchronize(ws->stream); ws->collect_spans(); }
      for (int i = 0; i < S3D_N_STAGES; ++i) {
        ctx->stage_ms[i] += ws->stage_ms[i]; ctx->stage_launches[i] += ws->stage_launches[i];
        ws->stage_ms[i] = 0; ws->stage_launches[i] = 0;
      }
    }
    std::lock_guard<std::mutex> g(dc->mu);
    dc->pool.push_back(std::move(ws));
  }
  Workspace& operator*() { return *ws; }
};

// Runs `body` (which sets up and processes one batch on `ws`); if the NN grid overflowed its optimistic hash arena the
// batch is repeated once with exactly the size the device reported.
template <typename F>
static void with_arena_retry(Workspace& ws, F&& body) {
  for (int attempt = 0;; ++attempt) {
    try {
      body();
      return;
    } catch (const ArenaOverflow& o) {
      cudaStreamSynchronize(ws.stream);
      ws.collect_spans();
      if (attempt >= 2) throw CudaError{"hash arena overflow persists after re-allocation"};
      ws.hash_want = o.needed;
    }
  }
}

template <typename F>
static int guarded(F&& f) {
  try {
    return f();
  } catch (const CudaError& e) {
    set_error(e.what);
    cudaGetLastError();
    return S3D_INTERNAL_ERROR;
  } catch (const std::exception& e) {
    set_error(e.what());
    return S3D_INTERNAL_ERROR;
  }
}

static void copy_out(Workspace& ws, void* dst, const void* src_dev, size_t bytes) {
  if (!dst || !bytes) return;
  S3D_CUDA(cudaMemcpyAsync(dst, src_dev, bytes, cudaMemcpyDefault, ws.stream));
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, dst) != cudaSuccess) { cudaGetLastError(); at.type = cudaMemoryTypeUnregistered; }
  if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) ws.d2h += bytes;
}

static void align_chunk_body(Workspace& ws, const std::vector<const float*>& clouds, const std::vector<uint64_t>& sizes, const double* guesses,
                             const s3d_registration_parameters& cfg, int n, s3d_result* out);

// One sub-batch of align() calls on one device.  With `fine` set, the chunk runs createConstraint's loop-closure sequence
// (PointCloudSensor.cpp:286-292): align with `cfg` (coarse), then align again with `fine` and the coarse result as the guess;
// the scans are uploaded once and the second pass reads them from the device staging buffer.
static void align_chunk(s3d_context* ctx, int slot, const s3d_cloud* sources, const s3d_cloud* targets, const double* guesses,
                        const s3d_registration_parameters& cfg, int n, s3d_result* out, const s3d_registration_parameters* fine = nullptr,
                        s3d_result* out_fine = nullptr) {
  WsLease lease(ctx, slot);
  Workspace& ws = *lease;
  std::vector<const float*> clouds(2 * n);
  std::vector<uint64_t> sizes(2 * n);
  for (int i = 0; i < n; ++i) {
    clouds[2 * i] = sources[i].xyzw; sizes[2 * i] = sources[i].n;
    clouds[2 * i + 1] = targets[i].xyzw; sizes[2 * i + 1] = targets[i].n;
  }
  with_arena_retry(ws, [&] { align_chunk_body(ws, clouds, sizes, guesses, cfg, n, out); });
  if (!fine) return;
  // second pass: every slot's raw points already sit on the device (user device memory or the staging buffer)
  SlotInfo* hs = ws.h_slots.as<SlotInfo>();
  std::vector<const float*> dev(2 * n);
  for (int s = 0; s < 2 * n; ++s) dev[s] = sizes[s] ? reinterpret_cast<const float*>(hs[s].raw) : nullptr;
  std::vector<double> g2(16 * (size_t)n);
  for (int i = 0; i < n; ++i) memcpy(&g2[16 * (size_t)i], out[i].T, sizeof(double) * 16);
  with_arena_retry(ws, [&] { align_chunk_body(ws, dev, sizes, g2.data(), *fine, n, out_fine); });
  for (int i = 0; i < n; ++i)
    if (out[i].status != S3D_OK) {  // the coarse align threw: createConstraint never reaches the fine align (:286-289)
      out_fine[i] = out[i];
    }
}

// GICP_OMP / NDT_OMP (PointCloudSensor.cpp:149-157) are pclomp's multi-threaded builds of the two algorithms — same
// objective, same optimiser, same parameters — so on the GPU path they select the GICP / NDT branch (SURVEY 8f-4).  NDT_OMP
// differs in one step, the neighbour search: ndt_direct7() says which one the branch runs.  Building with
// -DS3D_OMP_UNAVAILABLE keeps the behaviour of a reference build without pclomp (:158-161: std::runtime_error).
static int effective_algorithm(int alg) {
#ifndef S3D_OMP_UNAVAILABLE
  if (alg == S3D_ALG_GICP_OMP) return S3D_ALG_GICP;
  if (alg == S3D_ALG_NDT_OMP) return S3D_ALG_NDT;
#endif
  return alg;
}

// pclomp's NDT defaults to the DIRECT7 neighbour search and doNDT never changes it; PCL's NDT uses the kd-tree radius search.
// NDT_OMP runs DIRECT7 when the context selects it (s3d_set_ndt_omp_search); NDT always runs the radius search.
static bool ndt_direct7(const Workspace& ws, int requested_alg) {
  return effective_algorithm(requested_alg) == S3D_ALG_NDT && requested_alg == S3D_ALG_NDT_OMP && ws.ndt_omp_search == S3D_NDT_OMP_DIRECT7;
}

// S3D_TIMELINE=1 (measurement aid): device time stamps of a chunk's stages relative to one process-wide base event, printed
// to stderr after the chunk — the Gantt chart of the streams of a batch call (profiles/r02_summary.md).
struct Timeline {
  static bool enabled() { static const bool e = getenv("S3D_TIMELINE") != nullptr; return e; }
  static cudaEvent_t base(cudaStream_t st) {
    static std::mutex mu; static cudaEvent_t ev = nullptr;
    std::lock_guard<std::mutex> g(mu);
    if (!ev) { cudaEventCreate(&ev); cudaEventRecord(ev, st); }
    return ev;
  }
  cudaStream_t st; cudaEvent_t b; std::vector<std::pair<const char*, cudaEvent_t>> marks; int n;
  Timeline(Workspace& ws, int n_) : st(ws.stream), b(nullptr), n(n_) { if (enabled()) { b = base(st); mark("begin"); } }
  void mark(const char* what) { if (!b) return; cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); marks.emplace_back(what, e); }
  ~Timeline() {
    if (!b) return;
    std::string line = "[s3d timeline] stream " + std::to_string((unsigned long long)(uintptr_t)st % 100000) + " pairs " + std::to_string(n) + ":";
    for (auto& m : marks) { float ms = 0.f; cudaEventSynchronize(m.second); cudaEventElapsedTime(&ms, b, m.second); char buf[64]; snprintf(buf, sizeof buf, " %s %.3f", m.first, ms); line += buf; cudaEventDestroy(m.second); }
    fprintf(stderr, "%s\n", line.c_str());
  }
};

static void align_chunk_body(Workspace& ws, const std::vector<const float*>& clouds, const std::vector<uint64_t>& sizes, const double* guesses,
                             const s3d_registration_parameters& cfg_in, int n, s3d_result* out) {
  s3d_registration_parameters cfg = cfg_in;
  cfg.registration_algorithm = effective_algorithm(cfg_in.registration_algorithm);
  Timeline tl(ws, n);
  setup_batch(ws, clouds, sizes, n);
  tl.mark("setup");
  const float leaf = cfg.point_cloud_density > 0 ? (float)cfg.point_cloud_density : 0.f;  // :127, setLeafSize(float)
  run_voxel(ws, leaf);
  tl.mark("voxel");
  const bool gicp = cfg.registration_algorithm == S3D_ALG_GICP;
  const bool ndt = cfg.registration_algorithm == S3D_ALG_NDT;
  const bool k_ok = cfg.correspondence_randomness >= 1 && cfg.correspondence_randomness <= kMaxK;
  const bool ndt_ok = cfg.resolution > 0.f && std::isfinite(cfg.resolution);
  if (!(gicp && k_ok) && !(ndt && ndt_ok)) {
    // the reference evaluates the <100 gate before the algorithm switch (:134-135 then :139-165)
    SlotInfo* hs = ws.h_slots.as<SlotInfo>();
    S3D_CUDA(cudaMemcpyAsync(hs, ws.slots.p, sizeof(SlotInfo) * ws.n_slots, cudaMemcpyDeviceToHost, ws.stream));
    ws.sync();
    ws.d2h += sizeof(SlotInfo) * ws.n_slots;
    for (int i = 0; i < n; ++i) {
      memset(&out[i], 0, sizeof out[i]);
      for (int j = 0; j < 16; ++j) out[i].T[j] = (j % 5 == 0) ? 1.0 : 0.0;
      out[i].n_source = hs[2 * i].n_pts; out[i].n_target = hs[2 * i + 1].n_pts;
      if (out[i].n_source < 100 || out[i].n_target < 100) out[i].status = S3D_TOO_FEW_POINTS;
      else out[i].status = (gicp || ndt) ? S3D_INVALID_ARGUMENT : S3D_UNKNOWN_ALGORITHM;
    }
    if (gicp) set_error("correspondence_randomness must be in [1, 4096]");
    else if (ndt) set_error("NDT resolution must be positive");
    else if (cfg.registration_algorithm == S3D_ALG_GICP_OMP || cfg.registration_algorithm == S3D_ALG_NDT_OMP)
      set_error("OMP is not available, you need to rebuild SLAM3D with OMP or use another matching algorithm.");
    else set_error("Unknown registration algorithm specified.");
    return;
  }
  run_grid(ws, leaf);
  if (ndt) {  // doNDT  :84-117
    std::vector<s3d_registration_parameters> params(n, cfg);
    run_ndt(ws, params, guesses, ndt_direct7(ws, cfg_in.registration_algorithm), out);
    return;
  }
  tl.mark("grid");
  run_knn_covariances(ws, cfg.correspondence_randomness, nullptr, nullptr);
  tl.mark("knn");
  std::vector<s3d_registration_parameters> params(n, cfg);
  run_gicp(ws, params, guesses, out);
  tl.mark("gicp");
}

static const char* status_text(int st, const s3d_result& r, const s3d_registration_parameters& cfg, std::string& buf) {
  switch (st) {
    case S3D_TOO_FEW_POINTS: return "Too few points after filtering, you may have to decrease 'point_cloud_density'.";
    case S3D_NOT_CONVERGED:
      buf = std::string(cfg.registration_algorithm == S3D_ALG_NDT ? "NDT" : "ICP") + " failed with Fitness-Score " + std::to_string(r.fitness) + " > " +
            std::to_string(cfg.max_fitness_score);
      return buf.c_str();
    case S3D_TOO_FAR_FROM_GUESS: return "ICP result is to far away from guess";
    default: return nullptr;
  }
}

}  // namespace s3d

using namespace s3d;

extern "C" {

const char* s3d_last_error(void) { return g_last_error.c_str(); }
const char* s3d_version(void) { return "slam3d_b200 0.1 (sm_100a)"; }

void s3d_default_parameters(s3d_registration_parameters* p) {  // RegistrationParameters.hpp:36-97
  p->registration_algorithm = S3D_ALG_GICP;
  p->point_cloud_density = 0.2; p->max_fitness_score = 2.0; p->max_translation = 1.0; p->max_rotation = 1.0;
  p->euclidean_fitness_epsilon = 1.0; p->transformation_epsilon = 1e-5; p->max_correspondence_distance = 2.5;
  p->maximum_iterations = 50; p->rotation_epsilon = 2e-3; p->correspondence_randomness = 20; p->maximum_optimizer_iterations = 20;
  p->resolution = 1.0f; p->step_size = 0.05; p->outlier_ratio = 0.35;
}

int s3d_create_context(const int* devices, int n_devices, s3d_context** out) {
  if (!out) return S3D_INVALID_ARGUMENT;
  *out = nullptr;
  return guarded([&]() -> int {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
      cudaGetLastError();
      set_error("no CUDA device: the slam3d_b200 scan-matching path has no CPU fallback");
      return S3D_INTERNAL_ERROR;
    }
    std::unique_ptr<s3d_context> ctx(new s3d_context());
    std::vector<int> devs;
    if (devices && n_devices > 0) devs.assign(devices, devices + n_devices);
    else { int cur = 0; S3D_CUDA(cudaGetDevice(&cur)); devs.push_back(cur); }
    for (int d : devs) {
      if (d < 0 || d >= count) { set_error("bad device ordinal"); return S3D_INVALID_ARGUMENT; }
      std::unique_ptr<DeviceCtx> dc(new DeviceCtx());
      dc->device = d;
      std::unique_ptr<Workspace> ws(new Workspace());
      ws->init(d);
      dc->all.push_back(ws.get());
      dc->pool.push_back(std::move(ws));
      ctx->devs.push_back(std::move(dc));
    }
    if (const char* env = getenv("S3D_MAX_PAIRS_PER_LAUNCH")) ctx->max_pairs_per_launch = std::max(1, atoi(env));
    if (const char* env = getenv("S3D_STREAMS_PER_DEVICE")) ctx->streams_per_device = ctx->streams_small = std::max(1, atoi(env));
    *out = ctx.release();
    return S3D_OK;
  });
}

int s3d_destroy_context(s3d_context* ctx) {
  if (!ctx) return S3D_OK;
  for (auto& dc : ctx->devs) {
    for (auto& ws : dc->pool) ws->destroy();
    dc->pool.clear();
    cudaSetDevice(dc->device);
    for (auto& b : dc->free_blocks) cudaFree(b.first);
    dc->free_blocks.clear();
  }
  delete ctx;
  return S3D_OK;
}

void* s3d_context_stream(s3d_context* ctx, int device_slot) {
  if (!ctx || device_slot < 0 || device_slot >= (int)ctx->devs.size()) return nullptr;
  DeviceCtx* dc = ctx->devs[device_slot].get();
  std::lock_guard<std::mutex> g(dc->mu);
  return dc->all.empty() ? nullptr : (void*)dc->all[0]->stream;
}

int s3d_set_input_stream(s3d_context* ctx, void* stream, int enabled) {
  if (!ctx) return S3D_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(ctx->mu);
  ctx->input_stream = static_cast<cudaStream_t>(stream);
  ctx->have_input_stream = enabled != 0;
  return S3D_OK;
}

int s3d_set_gicp_optimizer(s3d_context* ctx, int optimizer, int* previous) {
  if (!ctx) return S3D_INVALID_ARGUMENT;
  if (optimizer != S3D_GICP_NEWTON && optimizer != S3D_GICP_BFGS) {
    set_error("GICP optimizer must be S3D_GICP_NEWTON (0) or S3D_GICP_BFGS (1)");
    return S3D_INVALID_ARGUMENT;
  }
  const int old = ctx->gicp_optimizer.exchange(optimizer);
  if (previous) *previous = old;
  return S3D_OK;
}

int s3d_set_ndt_omp_search(s3d_context* ctx, int method, int* previous) {
  if (!ctx) return S3D_INVALID_ARGUMENT;
  if (method != S3D_NDT_OMP_KDTREE && method != S3D_NDT_OMP_DIRECT7) {
    set_error("NDT_OMP search must be S3D_NDT_OMP_KDTREE (0) or S3D_NDT_OMP_DIRECT7 (1)");
    return S3D_INVALID_ARGUMENT;
  }
  const int old = ctx->ndt_omp_search.exchange(method);
  if (previous) *previous = old;
  return S3D_OK;
}

int s3d_get_counters(s3d_context* ctx, s3d_counters* out) {
  if (!ctx || !out) return S3D_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(ctx->mu);
  out->kernel_launches = ctx->launches; out->h2d_bytes = ctx->h2d; out->d2h_bytes = ctx->d2h;
  return S3D_OK;
}

int s3d_get_loop_stats(s3d_context* ctx, uint64_t* tiles, uint64_t* control_steps, int reset) {
  if (!ctx) return S3D_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (tiles) *tiles = ctx->loop_tiles;
  if (control_steps) *control_steps = ctx->loop_ctrl_steps;
  if (reset) ctx->loop_tiles = ctx->loop_ctrl_steps = 0;
  return S3D_OK;
}

int s3d_set_profiling(s3d_context* ctx, int enabled) {
  if (!ctx) return S3D_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(ctx->mu);
  ctx->profiling = enabled != 0;
  return S3D_OK;
}

int s3d_get_stage_times(s3d_context* ctx, double ms[S3D_N_STAGES], uint64_t launches[S3D_N_STAGES], int reset) {
  if (!ctx) return S3D_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(ctx->mu);
  for (int i = 0; i < S3D_N_STAGES; ++i) {
    if (ms) ms[i] = ctx->stage_ms[i];
    if (launches) launches[i] = ctx->stage_launches[i];
    if (reset) { ctx->stage_ms[i] = 0; ctx->stage_launches[i] = 0; }
  }
  return S3D_OK;
}

int s3d_voxel_downsample(s3d_context* ctx, s3d_cloud in, float leaf, float* out_xyzw, uint64_t* n_out, uint32_t* leaf_index, int32_t* overflow) {
  if (!ctx || !n_out) return S3D_INVALID_ARGUMENT;
  if (!(leaf > 0.f)) { set_error("leaf size must be positive"); return S3D_INVALID_ARGUMENT; }
  *n_out = 0;
  if (overflow) *overflow = 0;
  if (in.n == 0) return S3D_OK;  // PointCloudSensor.cpp:193
  return guarded([&]() -> int {
    WsLease lease(ctx, 0);
    Workspace& ws = *lease;
    setup_batch(ws, {in.xyzw}, {in.n}, 0);
    DevBuf& lk = ws.moved;  // borrowed as the unsorted-key buffer
    if (leaf_index) lk.reserve(4 * size_t(ws.total));
    run_voxel(ws, leaf, leaf_index ? lk.as<uint32_t>() : nullptr);
    SlotInfo* hs = ws.h_slots.as<SlotInfo>();
    S3D_CUDA(cudaMemcpyAsync(hs, ws.slots.p, sizeof(SlotInfo), cudaMemcpyDeviceToHost, ws.stream));
    ws.sync();
    ws.d2h += sizeof(SlotInfo);
    *n_out = hs[0].n_pts;
    if (overflow) *overflow = hs[0].overflow;
    copy_out(ws, out_xyzw, ws.work.p, 16 * size_t(hs[0].n_pts));
    copy_out(ws, leaf_index, lk.p, 4 * size_t(in.n));
    ws.sync();
    return S3D_OK;
  });
}

int s3d_knn_covariances(s3d_context* ctx, s3d_cloud cloud, int k, uint32_t* knn_index, float* knn_dist2, double* covariances) {
  if (!ctx) return S3D_INVALID_ARGUMENT;
  if (k < 1 || k > kMaxK || (uint64_t)k > cloud.n) { set_error("k must be in [1, 4096] and not larger than the cloud"); return S3D_INVALID_ARGUMENT; }
  return guarded([&]() -> int {
    WsLease lease(ctx, 0);
    Workspace& ws = *lease;
    int rc = S3D_OK;
    with_arena_retry(ws, [&] {
    setup_batch(ws, {cloud.xyzw}, {cloud.n}, 0);
    run_voxel(ws, 0.f);
    run_grid(ws, 0.f);
    const size_t n = cloud.n;
    DevBuf& di = ws.moved; DevBuf& dd = ws.prev_nn; DevBuf& dc = ws.moments;
    if (knn_index) di.reserve(4 * n * k);
    if (knn_dist2) dd.reserve(4 * n * k);
    run_knn_covariances(ws, k, knn_index ? di.as<uint32_t>() : nullptr, knn_dist2 ? dd.as<float>() : nullptr);
    if (covariances) { dc.reserve(72 * n); run_expand_cov(ws, dc.as<double>()); }
    int32_t* hf = ws.h_small.as<int32_t>();
    S3D_CUDA(cudaMemcpyAsync(hf, ws.flags.p, 16, cudaMemcpyDeviceToHost, ws.stream));
    ws.sync();
    check_arena(ws, hf);
    copy_out(ws, knn_index, di.p, 4 * n * k);
    copy_out(ws, knn_dist2, dd.p, 4 * n * k);
    copy_out(ws, covariances, dc.p, 72 * n);
    ws.sync();
    });
    return rc;
  });
}

int s3d_nearest_neighbors(s3d_context* ctx, s3d_cloud reference, s3d_cloud queries, const double* transform, uint32_t* nn_index, float* nn_dist2) {
  if (!ctx || reference.n == 0) return S3D_INVALID_ARGUMENT;
  if (queries.n == 0) return S3D_OK;
  return guarded([&]() -> int {
    WsLease lease(ctx, 0);
    Workspace& ws = *lease;
    with_arena_retry(ws, [&] {
    setup_batch(ws, {reference.xyzw, queries.xyzw}, {reference.n, queries.n}, 0);
    run_voxel(ws, 0.f);
    run_grid(ws, 0.f);
    float* Td = nullptr;
    if (transform) {
      float* hT = ws.h_small.as<float>() + 64;
      for (int i = 0; i < 16; ++i) hT[i] = (float)transform[i];
      ws.fit_partial.reserve(64);
      Td = ws.fit_partial.as<float>();
      S3D_CUDA(cudaMemcpyAsync(Td, hT, 64, cudaMemcpyHostToDevice, ws.stream));
    }
    DevBuf& di = ws.moved; DevBuf& dd = ws.prev_nn;
    di.reserve(4 * queries.n); dd.reserve(4 * queries.n);
    run_nn_stage(ws, 0, 1, Td, di.as<uint32_t>(), dd.as<float>());
    int32_t* hf = ws.h_small.as<int32_t>();
    S3D_CUDA(cudaMemcpyAsync(hf, ws.flags.p, 16, cudaMemcpyDeviceToHost, ws.stream));
    ws.sync();
    check_arena(ws, hf);
    copy_out(ws, nn_index, di.p, 4 * queries.n);
    copy_out(ws, nn_dist2, dd.p, 4 * queries.n);
    ws.sync();
    });
    return S3D_OK;
  });
}

// ---- per-measurement device cache ---------------------------------------------------------------------------------
static void* block_alloc(DeviceCtx* dc, size_t bytes, size_t* got) {
  {
    std::lock_guard<std::mutex> g(dc->mu);
    for (size_t i = 0; i < dc->free_blocks.size(); ++i)
      if (dc->free_blocks[i].second >= bytes && dc->free_blocks[i].second <= 2 * bytes + 4096) {
        void* p = dc->free_blocks[i].first; *got = dc->free_blocks[i].second;
        dc->free_blocks.erase(dc->free_blocks.begin() + i);
        ++dc->blocks_reused;
        return p;
      }
  }
  void* p = nullptr;
  S3D_CUDA(cudaMalloc(&p, bytes));
  *got = bytes;
  std::lock_guard<std::mutex> g(dc->mu);
  ++dc->blocks_allocated;
  return p;
}

namespace s3d {
// Per-cloud stages for `n` clouds in one workspace pass, then one device block per cloud.  resolution > 0 builds NDT handles
// (VoxelGridCovariance at `resolution`), otherwise GICP handles (kNN-k covariances and normals).
static void prepare_chunk(s3d_context* ctx, int device_slot, const s3d_cloud* clouds, int n, double density, int k, float resolution,
                          s3d_prepared_cloud** out) {
  WsLease lease(ctx, device_slot);
  Workspace& ws = *lease;
  const bool ndt = resolution > 0.f;
  const float leaf = density > 0 ? (float)density : 0.f;
  std::vector<const float*> ptrs(n);
  std::vector<uint64_t> sizes(n);
  uint64_t total = 0;
  for (int i = 0; i < n; ++i) { ptrs[i] = clouds[i].xyzw; sizes[i] = clouds[i].n; total += clouds[i].n; }
  SlotInfo* hs = nullptr;
  NdtGrid* hg = nullptr;
  with_arena_retry(ws, [&] {
    setup_batch(ws, ptrs, sizes, 0);
    run_voxel(ws, leaf);
    if (total) {
      run_grid(ws, leaf);
      if (ndt) {
        const std::vector<float> res(n, resolution);
        run_ndt_grids(ws, kNdtEverySlot, (uint32_t)n, res.data());
      } else {
        run_knn_covariances(ws, k, nullptr, nullptr);
      }
    }
    hs = ws.h_slots.as<SlotInfo>();
    int32_t* hf = ws.h_small.as<int32_t>();
    S3D_CUDA(cudaMemcpyAsync(hs, ws.slots.p, sizeof(SlotInfo) * n, cudaMemcpyDeviceToHost, ws.stream));
    S3D_CUDA(cudaMemcpyAsync(hf, ws.flags.p, 16, cudaMemcpyDeviceToHost, ws.stream));
    ws.d2h += sizeof(SlotInfo) * n + 16;
    if (ndt && total) {  // the grid sizes, which size the blocks, arrive with the same synchronise
      hg = ws.h_grids.as<NdtGrid>();
      S3D_CUDA(cudaMemcpyAsync(hg, ws.ndt_grids.p, sizeof(NdtGrid) * n, cudaMemcpyDeviceToHost, ws.stream));
      ws.d2h += sizeof(NdtGrid) * n;
    }
    ws.sync();
    ws.collect_spans();
    check_arena(ws, hf);
    ws.learn_grid_frac(hs, (uint32_t)n);
  });
  auto up = [](size_t b) { return (b + 255) & ~size_t(255); };
  std::vector<std::unique_ptr<s3d_prepared_cloud>> hh(n);
  struct BlockGuard {  // a failure below (allocation, copy, synchronise) hands the device blocks back instead of leaking them
    std::vector<std::unique_ptr<s3d_prepared_cloud>>& hh; DeviceCtx* dc; bool armed = true;
    ~BlockGuard() {
      if (!armed) return;
      std::lock_guard<std::mutex> g(dc->mu);
      for (auto& h : hh) if (h && h->block) { dc->free_blocks.emplace_back(h->block, h->block_bytes); h->block = nullptr; }
    }
  } guard{hh, ctx->devs[device_slot].get()};
  for (int i = 0; i < n; ++i) {
    std::unique_ptr<s3d_prepared_cloud>& h = hh[i];
    h.reset(new s3d_prepared_cloud());
    h->device_slot = device_slot; h->density = density; h->k = ndt ? 0 : k; h->resolution = ndt ? resolution : 0.f;
    h->info = hs[i];
    const size_t np = h->info.n_pts;
    if (ndt) {  // a cloud without a searchable grid (no finite point, int32 guard) keeps an empty one: its align ends at once
      if (hg) h->grid = hg[i];
      h->grid.resolution = resolution;
      h->grid.leaves = nullptr; h->grid.table = nullptr;
    }
    const size_t b_pts = up(16 * np), b_nrm = ndt ? 0 : up(32 * np), b_tab = up(sizeof(HashEntry) * (size_t)h->info.hash_cap);
    const bool ndt_arrays = ndt && h->grid.searchable;
    const size_t b_leaf = ndt_arrays ? up(sizeof(NdtLeaf) * (size_t)h->grid.n_voxels) : 0;
    const size_t b_ndt_tab = ndt_arrays ? up(sizeof(uint2) * ((size_t)h->grid.hash_mask + 1)) : 0;
    if (np) {
      h->block = block_alloc(ctx->devs[device_slot].get(), b_pts + b_nrm + b_tab + b_leaf + b_ndt_tab, &h->block_bytes);
      char* base = static_cast<char*>(h->block);
      S3D_CUDA(cudaMemcpyAsync(base, ws.gpts.as<float4>() + hs[i].off, 16 * np, cudaMemcpyDeviceToDevice, ws.stream));
      if (!ndt) S3D_CUDA(cudaMemcpyAsync(base + b_pts, ws.normals.as<double4>() + hs[i].off, 32 * np, cudaMemcpyDeviceToDevice, ws.stream));
      S3D_CUDA(cudaMemcpyAsync(base + b_pts + b_nrm, ws.hash.as<HashEntry>() + hs[i].hash_off, sizeof(HashEntry) * (size_t)h->info.hash_cap,
                               cudaMemcpyDeviceToDevice, ws.stream));
      h->info.gpts = reinterpret_cast<const float4*>(base);
      h->info.normals = ndt ? nullptr : reinterpret_cast<const double4*>(base + b_pts);
      h->info.table = reinterpret_cast<const HashEntry*>(base + b_pts + b_nrm);
      if (ndt_arrays) {  // leaf ranks in the hash are relative to the leaf array: copying both keeps them valid
        char* leaves = base + b_pts + b_tab;
        S3D_CUDA(cudaMemcpyAsync(leaves, hg[i].leaves, sizeof(NdtLeaf) * (size_t)h->grid.n_voxels, cudaMemcpyDeviceToDevice, ws.stream));
        S3D_CUDA(cudaMemcpyAsync(leaves + b_leaf, hg[i].table, sizeof(uint2) * ((size_t)h->grid.hash_mask + 1), cudaMemcpyDeviceToDevice, ws.stream));
        h->grid.leaves = reinterpret_cast<NdtLeaf*>(leaves);
        h->grid.table = reinterpret_cast<uint2*>(leaves + b_leaf);
      }
    } else {
      h->info.gpts = nullptr; h->info.normals = nullptr; h->info.table = nullptr; h->info.hash_cap = 0;
    }
    h->info.hash_off = 0; h->info.off = 0; h->info.raw = nullptr;
  }
  ws.sync();
  guard.armed = false;
  for (int i = 0; i < n; ++i) out[i] = hh[i].release();
}

// s3d_prepare_clouds / s3d_prepare_clouds_ndt: chunks of the n clouds on `streams_small` worker threads, all-or-nothing
static int prepare_clouds(s3d_context* ctx, int device_slot, const s3d_cloud* clouds, int n, double density, int k, float resolution,
                          s3d_prepared_cloud** out) {
  const int W = std::max(1, ctx->streams_small);
  const int chunk = balanced_chunk(n, W, 2 * ctx->max_pairs_per_launch);
  std::vector<int> st(W, S3D_OK);
  std::vector<std::string> errs(W);
  std::atomic<int> next{0};
  const bool threaded = !(W == 1 || n <= 2);
  auto worker = [&](int w) {
    t_gate_uploads = threaded; t_blocking_sync = threaded;
    g_last_error.clear();
    st[w] = guarded([&]() -> int {
      for (;;) {
        const int b = next.fetch_add(1) * chunk;
        if (b >= n) break;
        prepare_chunk(ctx, device_slot, clouds + b, std::min(chunk, n - b), density, k, resolution, out + b);
      }
      return S3D_OK;
    });
    errs[w] = g_last_error;
    t_gate_uploads = false; t_blocking_sync = false;
  };
  if (!threaded) worker(0);
  else ctx->parallel(W, worker);
  for (int w = 0; w < W; ++w)
    if (st[w] != S3D_OK) {
      for (int i = 0; i < n; ++i) { s3d_release_cloud(ctx, out[i]); out[i] = nullptr; }
      set_error(errs[w]);
      return st[w];
    }
  return S3D_OK;
}
}  // namespace s3d

int s3d_prepare_clouds(s3d_context* ctx, int device_slot, const s3d_cloud* clouds, int n, double density, int k, s3d_prepared_cloud** out) {
  if (!ctx || !out || n < 0 || (n > 0 && !clouds) || device_slot < 0 || device_slot >= (int)ctx->devs.size()) return S3D_INVALID_ARGUMENT;
  for (int i = 0; i < n; ++i) out[i] = nullptr;
  if (k < 1 || k > kMaxK) { set_error("correspondence_randomness must be in [1, 4096]"); return S3D_INVALID_ARGUMENT; }
  if (n == 0) return S3D_OK;
  return prepare_clouds(ctx, device_slot, clouds, n, density, k, 0.f, out);
}

int s3d_prepare_cloud(s3d_context* ctx, int device_slot, s3d_cloud cloud, double density, int k, s3d_prepared_cloud** out) {
  if (!out) return S3D_INVALID_ARGUMENT;
  return s3d_prepare_clouds(ctx, device_slot, &cloud, 1, density, k, out);
}

int s3d_prepare_clouds_ndt(s3d_context* ctx, int device_slot, const s3d_cloud* clouds, int n, double density, float resolution,
                           s3d_prepared_cloud** out) {
  if (!ctx || !out || n < 0 || (n > 0 && !clouds)) return S3D_INVALID_ARGUMENT;
  for (int i = 0; i < n; ++i) out[i] = nullptr;
  if (device_slot < 0 || device_slot >= (int)ctx->devs.size()) { set_error("bad device slot"); return S3D_INVALID_ARGUMENT; }
  if (!(resolution > 0.f) || !std::isfinite(resolution)) { set_error("NDT resolution must be positive and finite"); return S3D_INVALID_ARGUMENT; }
  if (std::isnan(density)) { set_error("point_cloud_density must not be NaN"); return S3D_INVALID_ARGUMENT; }
  if (n == 0) return S3D_OK;
  return prepare_clouds(ctx, device_slot, clouds, n, density, 0, resolution, out);
}

int s3d_prepare_cloud_ndt(s3d_context* ctx, int device_slot, s3d_cloud cloud, double density, float resolution, s3d_prepared_cloud** out) {
  if (!out) return S3D_INVALID_ARGUMENT;
  return s3d_prepare_clouds_ndt(ctx, device_slot, &cloud, 1, density, resolution, out);
}

int s3d_release_cloud(s3d_context* ctx, s3d_prepared_cloud* cloud) {
  if (!cloud) return S3D_OK;
  if (!ctx || cloud->device_slot >= (int)ctx->devs.size()) return S3D_INVALID_ARGUMENT;
  if (cloud->block) {
    DeviceCtx* dc = ctx->devs[cloud->device_slot].get();
    std::lock_guard<std::mutex> g(dc->mu);
    dc->free_blocks.emplace_back(cloud->block, cloud->block_bytes);  // recycled by the next prepare; freed with the context
  }
  delete cloud;
  return S3D_OK;
}

uint64_t s3d_prepared_cloud_size(const s3d_prepared_cloud* cloud) { return cloud ? cloud->info.n_pts : 0; }

int s3d_get_prepared_block_stats(s3d_context* ctx, uint64_t* allocated, uint64_t* reused) {
  if (!ctx) return S3D_INVALID_ARGUMENT;
  uint64_t a = 0, r = 0;
  for (auto& dc : ctx->devs) { std::lock_guard<std::mutex> g(dc->mu); a += dc->blocks_allocated; r += dc->blocks_reused; }
  if (allocated) *allocated = a;
  if (reused) *reused = r;
  return S3D_OK;
}

namespace s3d {
// One sub-batch of align() calls on prepared clouds (all on device slot `slot`).  GICP runs every pair; NDT runs the pairs whose
// fixed cloud (the source, slot 2p) is an NDT handle, and the others end as align() ends for an algorithm without its data.
static void align_prepared_chunk(s3d_context* ctx, int slot, const s3d_prepared_cloud* const* sources, const s3d_prepared_cloud* const* targets,
                                 const double* guesses, const s3d_registration_parameters& cfg_in, int n, s3d_result* out) {
  s3d_registration_parameters cfg = cfg_in;
  cfg.registration_algorithm = effective_algorithm(cfg_in.registration_algorithm);
  const bool gicp = cfg.registration_algorithm == S3D_ALG_GICP, ndt = cfg.registration_algorithm == S3D_ALG_NDT;
  std::vector<int> run;  // pairs that reach the optimiser, in batch order
  for (int i = 0; i < n; ++i) {
    if (gicp || (ndt && sources[i]->resolution > 0.f)) { run.push_back(i); continue; }
    // same order as align(): <100 gate first, then the algorithm switch
    memset(&out[i], 0, sizeof out[i]);
    for (int j = 0; j < 16; ++j) out[i].T[j] = (j % 5 == 0) ? 1.0 : 0.0;
    out[i].n_source = sources[i]->info.n_pts; out[i].n_target = targets[i]->info.n_pts;
    out[i].status = (out[i].n_source < 100 || out[i].n_target < 100) ? S3D_TOO_FEW_POINTS : S3D_UNKNOWN_ALGORITHM;
  }
  if ((int)run.size() < n) {
    if (cfg.registration_algorithm == S3D_ALG_GICP_OMP || cfg.registration_algorithm == S3D_ALG_NDT_OMP)
      set_error("OMP is not available, you need to rebuild SLAM3D with OMP or use another matching algorithm.");
    else if (ndt)
      set_error("NDT on prepared clouds needs the source scan prepared with s3d_prepare_clouds_ndt / s3d_prepare_cloud_ndt "
                "(this handle holds GICP data); or use s3d_gicp_align / s3d_gicp_align_batch on the raw clouds.");
    else set_error("Unknown registration algorithm specified.");
  }
  if (run.empty()) return;
  const int m = (int)run.size();
  WsLease lease(ctx, slot);
  Workspace& ws = *lease;
  S3D_CUDA(cudaSetDevice(ws.device));
  const uint32_t ns = 2 * m;
  ws.n_slots = ns; ws.n_pairs = m; ws.n_tiles = 0;
  ws.grid_frac = 1.f;  // prepared clouds: the sizes below are the filtered sizes
  ws.h_off.assign(ns, 0); ws.h_n.assign(ns, 0);
  ws.pair_off.resize(m);
  ws.slots.reserve(sizeof(SlotInfo) * ns);
  ws.h_slots.reserve(sizeof(SlotInfo) * ns);
  SlotInfo* hs = ws.h_slots.as<SlotInfo>();
  uint64_t total = 0;
  ws.max_na = 0;
  std::vector<double> g(16 * (size_t)m);
  std::vector<NdtGrid> grids(ndt ? m : 0);
  for (int j = 0; j < m; ++j) {
    const int i = run[j];
    hs[2 * j] = sources[i]->info; hs[2 * j + 1] = targets[i]->info;
    ws.h_n[2 * j] = sources[i]->info.n_pts; ws.h_n[2 * j + 1] = targets[i]->info.n_pts;
    ws.pair_off[j] = (uint32_t)total;
    total += (targets[i]->info.n_pts + 3u) & ~3u;
    ws.max_na = std::max(ws.max_na, targets[i]->info.n_pts);
    memcpy(&g[16 * (size_t)j], guesses + 16 * (size_t)i, sizeof(double) * 16);
    if (ndt) grids[j] = sources[i]->grid;
  }
  if (total >= (1ull << 31)) throw CudaError{"batch too large: more than 2^31 points"};
  ws.total = (uint32_t)total;
  S3D_CUDA(cudaMemcpyAsync(ws.slots.p, hs, sizeof(SlotInfo) * ns, cudaMemcpyHostToDevice, ws.stream));
  S3D_CUDA(cudaMemsetAsync(ws.flags.p, 0, 64, ws.stream));
  std::vector<s3d_registration_parameters> params(m, cfg);
  std::vector<s3d_result> res(m);
  if (ndt) run_ndt_prepared(ws, params, g.data(), grids.data(), ndt_direct7(ws, cfg_in.registration_algorithm), res.data());
  else run_gicp(ws, params, g.data(), res.data());
  for (int j = 0; j < m; ++j) out[run[j]] = res[j];
}
}  // namespace s3d

int s3d_gicp_align_prepared_batch(s3d_context* ctx, const s3d_prepared_cloud* const* sources, const s3d_prepared_cloud* const* targets,
                                  const double* guesses, const s3d_registration_parameters* params, int n_pairs, s3d_result* out) {
  if (!ctx || !params || !out || n_pairs < 0 || (n_pairs > 0 && (!sources || !targets || !guesses))) return S3D_INVALID_ARGUMENT;
  if (n_pairs == 0) return S3D_OK;
  const int slot = sources[0] ? sources[0]->device_slot : 0;
  const int alg = effective_algorithm(params->registration_algorithm);
  for (int i = 0; i < n_pairs; ++i) {
    if (!sources[i] || !targets[i]) return S3D_INVALID_ARGUMENT;
    if (sources[i]->device_slot != slot || targets[i]->device_slot != slot) { set_error("prepared clouds of one call must live on one device"); return S3D_INVALID_ARGUMENT; }
    for (const s3d_prepared_cloud* h : {sources[i], targets[i]})
      if (h->density != params->point_cloud_density || (alg == S3D_ALG_GICP && (h->k < 1 || h->k != params->correspondence_randomness))) {
        set_error(h->k < 1 && alg == S3D_ALG_GICP ? "prepared cloud holds NDT data (s3d_prepare_clouds_ndt): GICP needs s3d_prepare_clouds handles"
                                                  : "prepared cloud was built with another point_cloud_density / correspondence_randomness");
        return S3D_INVALID_ARGUMENT;
      }
    // NDT reads the source's grid (the PCL target) and the target's points only, so any handle of the right density serves as target
    float want = params->resolution, have = sources[i]->resolution;
    if (alg == S3D_ALG_NDT && have > 0.f && memcmp(&have, &want, sizeof(float)) != 0) {
      char buf[160];
      snprintf(buf, sizeof buf, "prepared cloud holds an NDT grid of resolution %.9g, the parameters ask for %.9g", (double)have, (double)want);
      set_error(buf);
      return S3D_INVALID_ARGUMENT;
    }
  }
  const int W = std::max(1, ctx->streams_small);
  std::vector<int> st(W, S3D_OK);
  std::vector<std::string> errs(W);
  std::atomic<int> next{0};
  const int chunk = balanced_chunk(n_pairs, W, ctx->max_pairs_per_launch);
  const bool threaded = !(W == 1 || n_pairs == 1);
  auto worker = [&](int w) {
    t_gate_uploads = threaded; t_blocking_sync = threaded;
    g_last_error.clear();
    st[w] = guarded([&]() -> int {
      for (;;) {
        const int b = next.fetch_add(1) * chunk;
        if (b >= n_pairs) break;
        const int n = std::min(chunk, n_pairs - b);
        align_prepared_chunk(ctx, slot, sources + b, targets + b, guesses + 16 * (size_t)b, *params, n, out + b);
      }
      return S3D_OK;
    });
    errs[w] = g_last_error;  // also the message of a per-pair status >= 4 inside a batch that ran (S3D_OK)
    t_gate_uploads = false; t_blocking_sync = false;
  };
  if (!threaded) worker(0);
  else ctx->parallel(W, worker);
  for (int w = 0; w < W; ++w) if (st[w] != S3D_OK) { set_error(errs[w]); return st[w]; }
  for (int w = 0; w < W; ++w) if (!errs[w].empty()) { set_error(errs[w]); break; }
  return S3D_OK;
}

int s3d_gicp_align_prepared(s3d_context* ctx, const s3d_prepared_cloud* source, const s3d_prepared_cloud* target, const double guess[16],
                            const s3d_registration_parameters* params, s3d_result* out) {
  if (!ctx || !params || !out || !guess || !source || !target) return S3D_INVALID_ARGUMENT;
  memset(out, 0, sizeof *out);
  const int st = s3d_gicp_align_prepared_batch(ctx, &source, &target, guess, params, 1, out);
  if (st != S3D_OK) { out->status = st; return st; }
  std::string buf;
  if (const char* msg = status_text(out->status, *out, *params, buf)) set_error(msg);
  return out->status;
}

// ---- patch and map building ------------------------------------------------------------------------------------------
int s3d_transform_cloud(s3d_context* ctx, s3d_cloud in, const double T[16], float* out_xyzw) {
  if (!ctx || !T || (in.n && !out_xyzw)) return S3D_INVALID_ARGUMENT;
  if (in.n == 0) return S3D_OK;
  return guarded([&]() -> int {
    WsLease lease(ctx, 0);
    Workspace& ws = *lease;
    const uint32_t n = run_accumulate(ws, {in.xyzw}, {in.n}, T);
    copy_out(ws, out_xyzw, ws.accu.p, 16 * (size_t)n);
    ws.sync();
    return S3D_OK;
  });
}

int s3d_create_combined_measurement(s3d_context* ctx, const s3d_cloud* clouds, const double* poses, int n, const double patch_pose[16],
                                    float* out_xyzw, uint64_t* n_out) {
  if (!ctx || !n_out || n < 0 || (n > 0 && (!clouds || !poses))) return S3D_INVALID_ARGUMENT;
  *n_out = 0;
  if (n == 0) return S3D_OK;
  return guarded([&]() -> int {
    WsLease lease(ctx, 0);
    Workspace& ws = *lease;
    std::vector<const float*> ptrs(n);
    std::vector<uint64_t> sizes(n);
    for (int i = 0; i < n; ++i) { ptrs[i] = clouds[i].xyzw; sizes[i] = clouds[i].n; }
    // pose.inverse() of an Eigen::Isometry3d: [R^T | -R^T t]
    double inv[16];
    if (patch_pose) {
      for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) inv[c * 4 + r] = patch_pose[r * 4 + c];
      for (int r = 0; r < 3; ++r) { double s = 0; for (int c = 0; c < 3; ++c) s += inv[c * 4 + r] * patch_pose[12 + c]; inv[12 + r] = -s; }
      inv[3] = inv[7] = inv[11] = 0; inv[15] = 1;
    }
    const uint32_t m = run_accumulate(ws, ptrs, sizes, poses, patch_pose ? inv : nullptr);
    if (m && !out_xyzw) return S3D_INVALID_ARGUMENT;
    copy_out(ws, out_xyzw, ws.accu.p, 16 * (size_t)m);
    ws.sync();
    *n_out = m;
    return S3D_OK;
  });
}

int s3d_remove_outliers(s3d_context* ctx, s3d_cloud in, double radius, unsigned min_neighbors, float* out_xyzw, uint64_t* n_out) {
  if (!ctx || !n_out || (in.n && !out_xyzw)) return S3D_INVALID_ARGUMENT;
  *n_out = 0;
  if (in.n == 0) return S3D_OK;
  return guarded([&]() -> int {
    WsLease lease(ctx, 0);
    Workspace& ws = *lease;
    const double I[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    ws.order_after_input();
    if (!(radius > 0 && min_neighbors > 0)) {  // :214 — the reference hands the input back
      S3D_CUDA(cudaMemcpyAsync(out_xyzw, in.xyzw, 16 * in.n, cudaMemcpyDefault, ws.stream));
      ws.sync();
      *n_out = in.n;
      return S3D_OK;
    }
    // stage the input on the device (identity transform would rewrite w; a plain copy keeps the points verbatim)
    ws.accu.reserve(16 * in.n); ws.accu2.reserve(16 * in.n);
    S3D_CUDA(cudaMemcpyAsync(ws.accu.p, in.xyzw, 16 * in.n, cudaMemcpyDefault, ws.stream));
    (void)I;
    uint32_t kept = 0;
    with_arena_retry(ws, [&] { kept = run_radius_filter(ws, ws.accu.as<float4>(), (uint32_t)in.n, radius, min_neighbors, ws.accu2.as<float4>()); });
    copy_out(ws, out_xyzw, ws.accu2.p, 16 * (size_t)kept);
    ws.sync();
    *n_out = kept;
    return S3D_OK;
  });
}

int s3d_build_map(s3d_context* ctx, const s3d_cloud* clouds, const double* poses, int n, double outlier_radius, unsigned outlier_neighbors,
                  double resolution, float* out_xyzw, uint64_t* n_out) {
  if (!ctx || !n_out || n < 0 || (n > 0 && (!clouds || !poses))) return S3D_INVALID_ARGUMENT;
  *n_out = 0;
  if (n == 0) return S3D_OK;
  return guarded([&]() -> int {
    WsLease lease(ctx, 0);
    Workspace& ws = *lease;
    std::vector<const float*> ptrs(n);
    std::vector<uint64_t> sizes(n);
    for (int i = 0; i < n; ++i) { ptrs[i] = clouds[i].xyzw; sizes[i] = clouds[i].n; }
    uint32_t m = run_accumulate(ws, ptrs, sizes, poses);                          // getAccumulatedCloud
    if (m == 0) return S3D_OK;
    const float4* cur = ws.accu.as<float4>();
    if (outlier_radius > 0 && outlier_neighbors > 0) {                             // removeOutliers
      ws.accu2.reserve(16 * (size_t)m);
      uint32_t kept = 0;
      with_arena_retry(ws, [&] { kept = run_radius_filter(ws, cur, m, outlier_radius, outlier_neighbors, ws.accu2.as<float4>()); });
      cur = ws.accu2.as<float4>(); m = kept;
    }
    if (m == 0) return S3D_OK;
    if (!(resolution > 0)) { set_error("map resolution must be positive"); return S3D_INVALID_ARGUMENT; }
    setup_batch(ws, {reinterpret_cast<const float*>(cur)}, {m}, 0);               // downsample
    run_voxel(ws, (float)resolution);
    SlotInfo* hs = ws.h_slots.as<SlotInfo>();
    S3D_CUDA(cudaMemcpyAsync(hs, ws.slots.p, sizeof(SlotInfo), cudaMemcpyDeviceToHost, ws.stream));
    ws.sync();
    ws.d2h += sizeof(SlotInfo);
    *n_out = hs[0].n_pts;
    copy_out(ws, out_xyzw, ws.work.p, 16 * (size_t)hs[0].n_pts);
    ws.sync();
    return S3D_OK;
  });
}

// ---- ground plane ------------------------------------------------------------------------------------------------------
namespace {
constexpr uint64_t kMaxGroundFill = (1ull << 31) - 1;

// the cloud in ws.accu (device): the sampler and the counting kernel read it many times, whatever memory it came from
const float4* stage_cloud(Workspace& ws, s3d_cloud cloud) {
  S3D_CUDA(cudaSetDevice(ws.device));
  ws.order_after_input();
  ws.accu.reserve(16 * cloud.n);
  S3D_CUDA(cudaMemcpyAsync(ws.accu.p, cloud.xyzw, 16 * cloud.n, cudaMemcpyDefault, ws.stream));
  return ws.accu.as<float4>();
}

int ransac_failed(const RansacFit& fit, uint64_t n) {
  if (n < 3) set_error("RANSAC plane fit: fewer than 3 points");
  else if (fit.iterations == 0) set_error("RANSAC plane fit: no non-degenerate sample of 3 points in 1000 draws");
  else set_error("RANSAC plane fit: no plane has an inlier");
  return S3D_INVALID_ARGUMENT;
}
}  // namespace

int s3d_fit_plane_ransac(s3d_context* ctx, s3d_cloud cloud, double threshold, int max_iterations, double probability,
                         float coefficients[4], int32_t* iterations, uint64_t* n_inliers, uint32_t* inliers) {
  if (!ctx || !coefficients || !iterations || !n_inliers || (cloud.n && !cloud.xyzw)) return S3D_INVALID_ARGUMENT;
  if (!(threshold > 0) || !std::isfinite(threshold) || !(probability > 0 && probability < 1) || max_iterations < 1) {
    set_error("RANSAC plane fit: threshold must be positive and finite, probability in (0, 1), max_iterations >= 1");
    return S3D_INVALID_ARGUMENT;
  }
  if (cloud.n >= (1ull << 31)) { set_error("RANSAC plane fit: more than 2^31 - 1 points"); return S3D_INVALID_ARGUMENT; }
  *iterations = 0; *n_inliers = 0;
  if (cloud.n < 3) return ransac_failed(RansacFit{}, cloud.n);
  return guarded([&]() -> int {
    WsLease lease(ctx, 0);
    Workspace& ws = *lease;
    const float4* pts = stage_cloud(ws, cloud);
    const RansacFit fit = run_ransac_plane(ws, pts, (uint32_t)cloud.n, threshold, max_iterations, probability, inliers != nullptr);
    *iterations = fit.iterations;
    if (!fit.ok) return ransac_failed(fit, cloud.n);
    for (int i = 0; i < 4; ++i) coefficients[i] = fit.coeff[i];
    *n_inliers = fit.n_inliers;
    if (inliers) { copy_out(ws, inliers, fit.inliers_dev, 4 * (size_t)fit.n_inliers); ws.sync(); }
    return S3D_OK;
  });
}

int s3d_ground_fill_size(double map_resolution, double radius, uint64_t* n) {
  if (!n) return S3D_INVALID_ARGUMENT;
  *n = 0;
  if (!(map_resolution > 0) || !(radius > 0) || !std::isfinite(map_resolution) || !std::isfinite(radius)) {
    set_error("ground fill: map resolution and radius must be positive and finite");
    return S3D_INVALID_ARGUMENT;
  }
  if (!ground_fill_lists(map_resolution, radius, kMaxGroundFill, nullptr, nullptr, nullptr, n)) {
    set_error("ground fill: more than 2^31 - 1 points");
    return S3D_INVALID_ARGUMENT;
  }
  return S3D_OK;
}

int s3d_fill_ground_plane(s3d_context* ctx, s3d_cloud cloud, double map_resolution, double radius, float* out_xyzw, float coefficients[4]) {
  uint64_t m = 0;
  if (!ctx || (cloud.n && !cloud.xyzw)) return S3D_INVALID_ARGUMENT;
  if (const int st = s3d_ground_fill_size(map_resolution, radius, &m)) return st;
  if (m && !out_xyzw) return S3D_INVALID_ARGUMENT;
  if (cloud.n >= (1ull << 31)) { set_error("ground fill: more than 2^31 - 1 points"); return S3D_INVALID_ARGUMENT; }
  if (cloud.n < 3) return ransac_failed(RansacFit{}, cloud.n);
  return guarded([&]() -> int {
    WsLease lease(ctx, 0);
    Workspace& ws = *lease;
    const float4* pts = stage_cloud(ws, cloud);
    const RansacFit fit = run_ransac_plane(ws, pts, (uint32_t)cloud.n, 0.01, 10000, 0.99, false);  // PointCloudSensor.cpp:364-366
    if (!fit.ok) return ransac_failed(fit, cloud.n);
    if (coefficients) for (int i = 0; i < 4; ++i) coefficients[i] = fit.coeff[i];
    std::vector<double> rings, sin_a, cos_a;
    uint64_t total = 0;
    ground_fill_lists(map_resolution, radius, kMaxGroundFill, &rings, &sin_a, &cos_a, &total);
    if (total == 0) return S3D_OK;
    ws.accu2.reserve(16 * total);
    run_ground_fill(ws, fit.coeff, rings, sin_a, cos_a, ws.accu2.as<float4>());
    copy_out(ws, out_xyzw, ws.accu2.p, 16 * total);
    ws.sync();  // the host vectors must outlive the copies
    return S3D_OK;
  });
}

static int align_batch_impl(s3d_context* ctx, const s3d_cloud* sources, const s3d_cloud* targets, const double* guesses,
                            const s3d_registration_parameters* params, int n_pairs, s3d_result* out, const s3d_registration_parameters* fine,
                            s3d_result* out_fine) {
  if (!ctx || !params || !out || n_pairs < 0 || (n_pairs > 0 && (!sources || !targets || !guesses))) return S3D_INVALID_ARGUMENT;
  if (n_pairs == 0) return S3D_OK;
  const int nd = (int)ctx->devs.size();
  // Contiguous shards, one per device; no device-to-device traffic (registrations are independent).  Inside a device the
  // shard is cut into chunks that `streams_per_device` host threads push through their own workspace/stream, so the H2D
  // copies and the per-iteration host polls of one chunk overlap with the kernels of another.
  const int W = std::max(1, params->registration_algorithm == S3D_ALG_NDT ? ctx->streams_small : ctx->streams_per_device);
  std::vector<int> st(nd * W, S3D_OK);
  std::vector<std::string> errs(nd * W);
  std::vector<std::atomic<int>> next(nd);
  for (auto& a : next) a.store(0);
  const bool threaded = !(nd * W == 1 || n_pairs == 1);
  auto worker = [&](int i) {
    const int d = i / W, w = i % W;
    const int lo = (int)((int64_t)n_pairs * d / nd), hi = (int)((int64_t)n_pairs * (d + 1) / nd);
    const int shard = hi - lo;
    if (shard <= 0) return;
    t_gate_uploads = threaded && W > 1; t_blocking_sync = threaded;
    g_last_error.clear();
    const int chunk = balanced_chunk(shard, W, ctx->max_pairs_per_launch);
    st[i] = guarded([&]() -> int {
      for (;;) {
        const int c = next[d].fetch_add(1);
        const int b = lo + c * chunk;
        if (b >= hi) break;
        const int n = std::min(chunk, hi - b);
        align_chunk(ctx, d, sources + b, targets + b, guesses + 16 * (size_t)b, *params, n, out + b, fine, fine ? out_fine + b : nullptr);
      }
      return S3D_OK;
    });
    errs[i] = g_last_error;  // also the message of a per-pair status >= 4 inside a batch that ran (S3D_OK)
    t_gate_uploads = false; t_blocking_sync = false;
  };
  if (!threaded) worker(0);
  else ctx->parallel(nd * W, worker);
  for (int i = 0; i < nd * W; ++i)
    if (st[i] != S3D_OK) { set_error(errs[i]); return st[i]; }
  for (int i = 0; i < nd * W; ++i) if (!errs[i].empty()) { set_error(errs[i]); break; }
  return S3D_OK;
}

int s3d_gicp_align_batch(s3d_context* ctx, const s3d_cloud* sources, const s3d_cloud* targets, const double* guesses,
                         const s3d_registration_parameters* params, int n_pairs, s3d_result* out) {
  return align_batch_impl(ctx, sources, targets, guesses, params, n_pairs, out, nullptr, nullptr);
}

int s3d_gicp_align_loop_batch(s3d_context* ctx, const s3d_cloud* sources, const s3d_cloud* targets, const double* guesses,
                              const s3d_registration_parameters* coarse, const s3d_registration_parameters* fine, int n_pairs,
                              s3d_result* out_coarse, s3d_result* out_fine) {
  if (!fine || !out_fine) return S3D_INVALID_ARGUMENT;
  std::vector<s3d_result> tmp;
  if (!out_coarse && n_pairs > 0) { tmp.resize(n_pairs); out_coarse = tmp.data(); }
  return align_batch_impl(ctx, sources, targets, guesses, coarse, n_pairs, out_coarse, fine, out_fine);
}

int s3d_gicp_align(s3d_context* ctx, s3d_cloud source, s3d_cloud target, const double guess[16], const s3d_registration_parameters* params,
                   s3d_result* out) {
  if (!ctx || !params || !out || !guess) return S3D_INVALID_ARGUMENT;
  memset(out, 0, sizeof *out);
  const int st = guarded([&]() -> int {
    align_chunk(ctx, 0, &source, &target, guess, *params, 1, out);
    return S3D_OK;
  });
  if (st != S3D_OK) { out->status = st; return st; }
  std::string buf;
  if (const char* msg = status_text(out->status, *out, *params, buf)) set_error(msg);
  return out->status;
}

}  // extern "C"
