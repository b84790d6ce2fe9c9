// voxel.cu — batch set-up and the VoxelGrid down-sampling kernels.
//
// Replaces pcl::VoxelGrid<PointXYZ>::filter as called from PointCloudSensor::downsample
// (slam3d/sensor/pcl/PointCloudSensor.cpp:190-201) and twice per align() (:127-131).  Semantics: SURVEY A.1.
//   bbox      min/max over finite points (ordered-uint atomics; min/max are order independent => deterministic)
//   params    per-slot scalars of A.1 steps 1,3,4 incl. the int32 overflow guard (one thread per slot)
//   keys      A.1 step 5, float ops in PCL's order via __fmul_rn/__fsub_rn (no FMA contraction)
//   sort      stable segmented radix sort (sort.cuh)                    A.1 step 6
//   heads     run starts -> per-tile counts -> per-slot scan           A.1 step 7
//   centroid  one thread per run sums its points in ascending input order in float, / float(count)   A.1 steps 8,9
// All kernels are streaming and HBM/L2-bandwidth bound: 16 B/point in, 8 B/point keys, 16 B/voxel out.
#include <atomic>
#include <condition_variable>
#include <deque>
#include <thread>

#include "internal.h"
#include "bbox.cuh"
#include "sort.cuh"

namespace s3d {

// ------------------------------------------------------------------------------------------------------------
void Workspace::init(int dev) {
  device = dev;
  S3D_CUDA(cudaSetDevice(dev));
  S3D_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev));
  S3D_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  S3D_CUDA(cudaEventCreateWithFlags(&sync_event, cudaEventBlockingSync | cudaEventDisableTiming));
  S3D_CUDA(cudaEventCreateWithFlags(&input_event, cudaEventDisableTiming));
  flags.reserve(64);
  h_small.reserve(4096);
}

// Single calls spin on the stream (lowest latency).  The chunks of a batch call run on several host threads per device — and
// under torchrun on several ranks per box — so they sleep on a blocking event instead: 8 ranks x 6 spinning threads on a
// 32-core host was the 8-GPU scaling loss of round 1.
void Workspace::sync() {
  if (blocking_sync && sync_event) {
    S3D_CUDA(cudaEventRecord(sync_event, stream));
    S3D_CUDA(cudaEventSynchronize(sync_event));
  } else {
    S3D_CUDA(cudaStreamSynchronize(stream));
  }
}

// device inputs produced on the caller's stream (s3d_set_input_stream): order this workspace's stream after it
void Workspace::order_after_input() {
  if (!wait_input) return;
  S3D_CUDA(cudaEventRecord(input_event, input_stream));
  S3D_CUDA(cudaStreamWaitEvent(stream, input_event, 0));
}

cudaEvent_t Workspace::get_event() {
  if (!event_pool.empty()) { cudaEvent_t e = event_pool.back(); event_pool.pop_back(); return e; }
  cudaEvent_t e;
  S3D_CUDA(cudaEventCreate(&e));
  return e;
}

void Workspace::collect_spans() {
  for (Span& sp : spans) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess) { stage_ms[sp.stage] += ms; stage_launches[sp.stage] += sp.n_launch; }
    else cudaGetLastError();
    event_pool.push_back(sp.a); event_pool.push_back(sp.b);
  }
  spans.clear();
}

void Workspace::destroy() {
  cudaSetDevice(device);
  if (stream) cudaStreamSynchronize(stream);
  collect_spans();
  for (cudaEvent_t e : event_pool) cudaEventDestroy(e);
  event_pool.clear();
  if (sync_event) cudaEventDestroy(sync_event);
  if (input_event) cudaEventDestroy(input_event);
  sync_event = input_event = nullptr;
  for (auto& g : loop_graphs) cudaGraphExecDestroy(g.second);
  for (cudaGraph_t g : loop_graph_defs) cudaGraphDestroy(g);
  loop_graphs.clear(); loop_graph_defs.clear();

  DevBuf* bufs[] = {&slots, &pairs, &raw_stage, &work, &gpts, &keys0, &keys1, &vals0, &vals1, &hist, &sort_totals, &long_runs, &tile_slot, &tile_first,
                    &slot_tile_begin, &tile_heads, &hash, &normals, &moved, &prev_nn, &sec_lb, &moments, &eval_part, &corr, &mahal, &iter_tile_pair, &iter_tile_first,
                    &fit_partial, &flags, &accu, &accu2, &map_aux, &ndt_pairs, &ndt_leaves, &ndt_hash, &ndt_part, &ndt_grids, &gicp_args, &gicp_sched, &knn_arena, &ransac, &ransac_idx};
  for (DevBuf* b : bufs) b->release();
  h_slots.release(); h_pairs.release(); h_small.release(); h_tiles.release(); h_grids.release(); h_bounce.release(); h_ransac.release();
  if (stream) cudaStreamDestroy(stream);
  stream = nullptr;
}

// ------------------------------------------------------------------------------------------------------------
// Pageable -> pinned staging copies, spread over a few helper threads shared by all workspaces of the process.  One thread's
// memcpy moves ~10 GB/s; a chunk of 16 scan pairs is 134 MB, so a chunk's own thread needed 13 ms for what its GPU work does in 5.
// Pieces of 1 MB go to a queue; the caller copies pieces too and returns when all of ITS pieces are done.
class CopyPool {
 public:
  static CopyPool& get() { static CopyPool p; return p; }
  struct Job { char* dst; const char* src; size_t bytes; std::atomic<int>* left; };
  void copy(const std::vector<std::pair<void*, std::pair<const void*, size_t>>>& spans) {
    constexpr size_t kPiece = 1u << 20;
    std::atomic<int> left{0};
    std::vector<Job> jobs;
    for (const auto& sp : spans)
      for (size_t o = 0; o < sp.second.second; o += kPiece)
        jobs.push_back(Job{static_cast<char*>(sp.first) + o, static_cast<const char*>(sp.second.first) + o, std::min(kPiece, sp.second.second - o), &left});
    if (jobs.empty()) return;
    left.store((int)jobs.size());
    if (n_threads_ > 0 && jobs.size() > 1) {
      { std::lock_guard<std::mutex> g(mu_); for (const Job& j : jobs) q_.push_back(j); }
      cv_.notify_all();
    } else {
      for (const Job& j : jobs) { memcpy(j.dst, j.src, j.bytes); }
      return;
    }
    for (;;) {  // help until the queue is empty, then wait for the pieces other threads still hold
      Job j;
      { std::lock_guard<std::mutex> g(mu_); if (q_.empty()) break; j = q_.front(); q_.pop_front(); }
      memcpy(j.dst, j.src, j.bytes);
      j.left->fetch_sub(1, std::memory_order_acq_rel);
    }
    while (left.load(std::memory_order_acquire) > 0) std::this_thread::yield();
  }
 private:
  CopyPool() {
    // helpers = half the cores this rank can count on (torchrun exports LOCAL_WORLD_SIZE), at most 8; S3D_COPY_THREADS overrides
    int n = (int)std::thread::hardware_concurrency();
    const char* lws = getenv("LOCAL_WORLD_SIZE");
    n = n / (2 * std::max(1, lws ? atoi(lws) : 1));
    n = std::min(8, std::max(0, n - 1));
    if (const char* e = getenv("S3D_COPY_THREADS")) n = std::max(0, atoi(e));
    n_threads_ = n;
    for (int i = 0; i < n; ++i) threads_.emplace_back([this] { loop(); });
  }
  ~CopyPool() {
    { std::lock_guard<std::mutex> g(mu_); stop_ = true; }
    cv_.notify_all();
    for (auto& t : threads_) t.join();
  }
  void loop() {
    std::unique_lock<std::mutex> lk(mu_);
    for (;;) {
      cv_.wait(lk, [this] { return stop_ || !q_.empty(); });
      if (stop_) return;
      Job j = q_.front(); q_.pop_front();
      lk.unlock();
      memcpy(j.dst, j.src, j.bytes);
      j.left->fetch_sub(1, std::memory_order_acq_rel);
      lk.lock();
    }
  }
  std::vector<std::thread> threads_;
  std::deque<Job> q_;
  std::mutex mu_;
  std::condition_variable cv_;
  int n_threads_ = 0;
  bool stop_ = false;
};

static cudaPointerAttributes pointer_attributes(const void* p) {
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); at.type = cudaMemoryTypeUnregistered; }
  return at;
}

// Pageable host clouds (a std::vector, the points of a pcl::PointCloud): cudaMemcpyAsync from pageable memory is staged by the
// driver through one small pinned buffer and blocks the calling thread (~10 GB/s, measured: e2e 1800 against 2430
// registrations/s from pinned memory).  The chunk's host thread copies them into the workspace's own pinned buffer instead —
// the host threads of the other chunks do the same in parallel, before they queue for the upload turn — and the DMA runs from there.
static bool pinned_bounce_enabled() {
  static const bool enabled = [] { const char* e = getenv("S3D_PINNED_BOUNCE"); return !e || atoi(e) != 0; }();  // 0: A/B measurements
  return enabled;
}

// s3d_upload_scans: verbatim copies of clouds[i] into dst[i] (device memory of ws.device), staged as setup_batch stages its inputs.
// Pageable clouds are copied in rounds of at most kRound bytes through the pinned bounce buffer, so it stays bounded however many
// scans one call uploads.  Host bytes count in ws.h2d; device clouds (of this or another GPU) are copied device to device.
void upload_clouds(Workspace& ws, const std::vector<const float*>& clouds, const std::vector<uint64_t>& sizes, const std::vector<float4*>& dst) {
  constexpr size_t kRound = size_t(256) << 20;
  S3D_CUDA(cudaSetDevice(ws.device));
  ws.order_after_input();
  const size_t n = clouds.size();
  std::vector<int> host(n, 0), via_bounce(n, 0);
  for (size_t i = 0; i < n; ++i) {
    if (!sizes[i]) continue;
    const cudaPointerAttributes at = pointer_attributes(clouds[i]);
    host[i] = at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged;
    via_bounce[i] = at.type == cudaMemoryTypeUnregistered && pinned_bounce_enabled();
  }
  std::vector<size_t> at_bounce(n, 0);  // offset of a pageable cloud in the bounce buffer during its round
  for (size_t b = 0; b < n;) {
    size_t e = b, pinned = 0;  // this round: clouds [b, e), `pinned` bytes of them through the bounce buffer
    std::vector<std::pair<void*, std::pair<const void*, size_t>>> spans;
    for (; e < n; ++e) {
      const size_t bytes = 16 * size_t(sizes[e]);
      if (!via_bounce[e]) continue;
      if (pinned && pinned + bytes > kRound) break;
      at_bounce[e] = pinned;
      pinned += bytes;
    }
    if (pinned) {
      ws.h_bounce.reserve(pinned);
      for (size_t i = b; i < e; ++i)
        if (via_bounce[i]) spans.push_back({ws.h_bounce.as<char>() + at_bounce[i], {clouds[i], 16 * size_t(sizes[i])}});
      CopyPool::get().copy(spans);
    }
    for (size_t i = b; i < e; ++i) {
      if (!sizes[i]) continue;
      const void* from = via_bounce[i] ? static_cast<const void*>(ws.h_bounce.as<char>() + at_bounce[i]) : static_cast<const void*>(clouds[i]);
      S3D_CUDA(cudaMemcpyAsync(dst[i], from, 16 * size_t(sizes[i]), cudaMemcpyDefault, ws.stream));
      if (host[i]) ws.h2d += 16 * size_t(sizes[i]);
    }
    ws.sync();  // the bounce buffer is refilled by the next round
    b = e;
  }
}

// ------------------------------------------------------------------------------------------------------------
// Batch set-up: slot table, tile table, input staging.  clouds[2p] = slam3d source of pair p, clouds[2p+1] = target
// (or any list of clouds for the stage-level entry points).
void setup_batch(Workspace& ws, const std::vector<const float*>& clouds, const std::vector<uint64_t>& sizes, uint32_t n_pairs) {
  S3D_CUDA(cudaSetDevice(ws.device));
  const uint32_t ns = static_cast<uint32_t>(clouds.size());
  ws.n_slots = ns; ws.n_pairs = n_pairs;
  ws.grid_frac = 1.f; ws.batch_leaf = 0.f;  // until run_voxel knows the leaf size
  ws.h_off.resize(ns); ws.h_n.resize(ns);
  uint64_t total = 0; uint32_t n_tiles = 0;
  for (uint32_t s = 0; s < ns; ++s) {
    ws.h_off[s] = static_cast<uint32_t>(total);
    ws.h_n[s] = static_cast<uint32_t>(sizes[s]);
    total += (sizes[s] + 3) & ~uint64_t(3);  // keep every slot 64-byte aligned
    n_tiles += static_cast<uint32_t>((sizes[s] + kSortTile - 1) / kSortTile);
  }
  if (total >= (1ull << 31)) throw CudaError{"batch too large: more than 2^31 points"};
  for (uint32_t s = 0; s < ns; ++s)
    if (sizes[s] >= (1ull << 30)) throw CudaError{"cloud too large: 2^30 points or more (the sort's look-back words count 30 bits)"};
  ws.total = static_cast<uint32_t>(total); ws.n_tiles = n_tiles;
  const size_t tot = std::max<size_t>(total, 4);
  ws.slots.reserve(sizeof(SlotInfo) * ns);
  ws.work.reserve(16 * tot); ws.gpts.reserve(16 * tot); ws.normals.reserve(32 * tot);
  // hash arena: ~1.2 occupied cells per point is typical for voxel-filtered lidar scans; 3 entries/point leaves 25% head-room
  // at load factor 1/2.  Sparse clouds (every point alone in its cell on many levels) overflow it: the layout kernel
  // then flags kErrHashArena and reports the exact need, and the caller re-runs the batch (with_arena_retry in api.cu).
  {
    const size_t want = std::max(ws.hash_want, 3 * size_t(total) + 64 * size_t(ns));
    if (ws.hash_cap < want) { ws.hash.reserve(sizeof(HashEntry) * want); ws.hash_cap = want; }
  }
  ws.pair_off.resize(n_pairs);
  ws.max_na = 0;
  for (uint32_t p = 0; p < n_pairs; ++p) { ws.pair_off[p] = ws.h_off[2 * p + 1]; ws.max_na = std::max(ws.max_na, ws.h_n[2 * p + 1]); }
  ws.keys0.reserve(4 * tot); ws.keys1.reserve(4 * tot); ws.vals0.reserve(4 * tot); ws.vals1.reserve(4 * tot);
  {
    const size_t words = 256 * size_t(std::max<uint32_t>(n_tiles, 1));
    if (words > ws.status_words) {  // new memory must not hold words that look like a current epoch
      ws.hist.reserve(sizeof(uint64_t) * words);
      ws.status_words = ws.hist.cap / sizeof(uint64_t);
      S3D_CUDA(cudaMemsetAsync(ws.hist.p, 0, ws.hist.cap, ws.stream));
    }
  }
  ws.sort_totals.reserve(sort_aux_bytes(std::max<uint32_t>(ns, 1)));
  ws.long_runs.reserve(sizeof(uint4) * (tot / 64 + ns + 1));
  ws.tile_slot.reserve(4 * std::max<uint32_t>(n_tiles, 1)); ws.tile_first.reserve(4 * std::max<uint32_t>(n_tiles, 1));
  ws.tile_heads.reserve(4 * std::max<uint32_t>(n_tiles, 1));
  ws.slot_tile_begin.reserve(4 * (ns + 1));
  ws.h_slots.reserve(sizeof(SlotInfo) * ns);
  ws.h_tiles.reserve(4 * (2 * size_t(n_tiles) + ns + 1));

  // classify input pointers; host memory (pinned or pageable), misaligned device memory and device memory of another GPU (a view
  // of a scan resident on one device inside a batch sharded over several) go through raw_stage
  bool need_stage = false, need_bounce = false;
  std::vector<int> on_device(ns, 0), pageable(ns, 0), other_device(ns, 0);
  for (uint32_t s = 0; s < ns; ++s) {
    if (sizes[s] == 0) continue;
    const cudaPointerAttributes at = pointer_attributes(clouds[s]);
    other_device[s] = at.type == cudaMemoryTypeDevice && at.device != ws.device;
    on_device[s] = (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) && !other_device[s] && (reinterpret_cast<uintptr_t>(clouds[s]) & 15) == 0;
    pageable[s] = at.type == cudaMemoryTypeUnregistered;
    if (!on_device[s]) need_stage = true;
    if (pageable[s]) need_bounce = true;
  }
  if (need_stage) ws.raw_stage.reserve(16 * tot);
  if (need_bounce && pinned_bounce_enabled()) {
    ws.h_bounce.reserve(16 * tot);
    std::vector<std::pair<void*, std::pair<const void*, size_t>>> spans;
    for (uint32_t s = 0; s < ns; ++s)
      if (pageable[s]) spans.push_back({ws.h_bounce.as<char>() + 16 * size_t(ws.h_off[s]), {clouds[s], 16 * size_t(sizes[s])}});
    CopyPool::get().copy(spans);
  } else {
    need_bounce = false;
  }

  ws.order_after_input();
  std::unique_lock<std::mutex> gate;  // uploads of concurrent chunks take turns (api.cu, t_gate_uploads)
  if (need_stage && ws.upload_gate) gate = std::unique_lock<std::mutex>(*ws.upload_gate);
  SlotInfo* hs = ws.h_slots.as<SlotInfo>();
  uint32_t* ht = ws.h_tiles.as<uint32_t>();
  uint32_t* h_tile_slot = ht; uint32_t* h_tile_first = ht + n_tiles; uint32_t* h_begin = ht + 2 * size_t(n_tiles);
  uint32_t t = 0;
  for (uint32_t s = 0; s < ns; ++s) {
    SlotInfo& si = hs[s];
    memset(&si, 0, sizeof si);
    si.off = ws.h_off[s]; si.n_raw = ws.h_n[s];
    si.gpts = ws.gpts.as<float4>() + si.off; si.normals = ws.normals.as<double4>() + si.off; si.table = ws.hash.as<HashEntry>();
    for (int a = 0; a < 3; ++a) {  // ordered-uint encodings of +inf / -inf, filled in by the bbox kernel
      reinterpret_cast<uint32_t&>(si.bb_min[a]) = 0xFFFFFFFFu; reinterpret_cast<uint32_t&>(si.bb_max[a]) = 0u;
      reinterpret_cast<uint32_t&>(si.g_min[a]) = 0xFFFFFFFFu; reinterpret_cast<uint32_t&>(si.g_max[a]) = 0u;
    }
    if (sizes[s] == 0) si.raw = nullptr;
    else if (on_device[s]) si.raw = reinterpret_cast<const float4*>(clouds[s]);
    else {
      si.raw = ws.raw_stage.as<float4>() + si.off;
      const void* from = (need_bounce && pageable[s]) ? static_cast<const void*>(ws.h_bounce.as<char>() + 16 * size_t(si.off)) : static_cast<const void*>(clouds[s]);
      S3D_CUDA(cudaMemcpyAsync(ws.raw_stage.as<float4>() + si.off, from, 16 * sizes[s], cudaMemcpyDefault, ws.stream));  // another GPU's memory: device to device
      if (!other_device[s]) ws.h2d += 16 * sizes[s];
    }
    h_begin[s] = t;
    for (uint64_t f = 0; f < sizes[s]; f += kSortTile) { h_tile_slot[t] = s; h_tile_first[t] = static_cast<uint32_t>(f); ++t; }
  }
  h_begin[ns] = t;
  if (gate.owns_lock()) { ws.sync(); gate.unlock(); }
  S3D_CUDA(cudaMemcpyAsync(ws.slots.p, hs, sizeof(SlotInfo) * ns, cudaMemcpyHostToDevice, ws.stream));
  if (n_tiles) {
    S3D_CUDA(cudaMemcpyAsync(ws.tile_slot.p, h_tile_slot, 4 * size_t(n_tiles), cudaMemcpyHostToDevice, ws.stream));
    S3D_CUDA(cudaMemcpyAsync(ws.tile_first.p, h_tile_first, 4 * size_t(n_tiles), cudaMemcpyHostToDevice, ws.stream));
  }
  S3D_CUDA(cudaMemcpyAsync(ws.slot_tile_begin.p, h_begin, 4 * size_t(ns + 1), cudaMemcpyHostToDevice, ws.stream));
  S3D_CUDA(cudaMemsetAsync(ws.flags.p, 0, 64, ws.stream));
}

// A.1 steps 1, 3, 4 — run per slot by the last CTA of the bbox launch (bbox.cuh).  leaf <= 0: no filtering, the working cloud is the raw cloud.
struct VoxelParams {
  float leaf;
  __device__ void operator()(SlotInfo& si) const {
    for (int a = 0; a < 3; ++a) {
      si.bb_min[a] = ordered_to_float(reinterpret_cast<uint32_t&>(si.bb_min[a]));
      si.bb_max[a] = ordered_to_float(reinterpret_cast<uint32_t&>(si.bb_max[a]));
    }
    if (!(leaf > 0.f)) { si.overflow = 1; si.n_pts = si.n_raw; return; }  // pass-through (treated like the overflow copy)
    if (si.n_finite == 0) { si.n_pts = 0; si.overflow = 0; return; }
    const float inv = __fdiv_rn(1.0f, leaf);
    si.inv_leaf = inv;
    const long long dx = (long long)__fmul_rn(__fsub_rn(si.bb_max[0], si.bb_min[0]), inv) + 1;
    const long long dy = (long long)__fmul_rn(__fsub_rn(si.bb_max[1], si.bb_min[1]), inv) + 1;
    const long long dz = (long long)__fmul_rn(__fsub_rn(si.bb_max[2], si.bb_min[2]), inv) + 1;
    if (dx * dy * dz > 2147483647ll) { si.overflow = 1; si.n_pts = si.n_raw; return; }  // "output = *input_"
    int div_b[3];
    for (int a = 0; a < 3; ++a) {
      si.min_b[a] = (int)floorf(__fmul_rn(si.bb_min[a], inv));
      const int max_b = (int)floorf(__fmul_rn(si.bb_max[a], inv));
      div_b[a] = max_b - si.min_b[a] + 1;
    }
    si.mul1 = (uint32_t)div_b[0];
    si.mul2 = (uint32_t)div_b[0] * (uint32_t)div_b[1];
    si.overflow = 0;
  }
};

// A.1 step 5
// + the digit totals of all four sort passes (sort.cuh), so that the sort never reads the keys just to count them
__global__ void __launch_bounds__(kSortThreads) voxel_keys_kernel(const SlotInfo* __restrict__ slots, TileMap tm, uint32_t n_slots, uint32_t* __restrict__ keys,
                                                                   uint32_t* __restrict__ totals) {
  __shared__ uint32_t sh[kSortPasses][256];
  const uint32_t t = blockIdx.x;
  const uint32_t slot = tm.tile_slot[t], first = tm.tile_first[t];
  const SlotInfo& si = slots[slot];
  if (si.overflow) return;
#pragma unroll
  for (int p = 0; p < kSortPasses; ++p) sh[p][threadIdx.x] = 0;
  __syncthreads();
  const float inv = si.inv_leaf;
  const float mb0 = (float)si.min_b[0], mb1 = (float)si.min_b[1], mb2 = (float)si.min_b[2];
#pragma unroll
  for (int j = 0; j < kSortTile / kSortThreads; ++j) {
    const uint32_t e = first + j * kSortThreads + threadIdx.x;
    if (e < si.n_raw) {
      const float4 v = __ldg(si.raw + e);  // the pointer comes out of the slot table: without __ldg the load is a generic LD
      uint32_t key = kInvalidKey;
      if (finite3(v.x, v.y, v.z)) {
        const int i0 = (int)__fsub_rn(floorf(__fmul_rn(v.x, inv)), mb0);
        const int i1 = (int)__fsub_rn(floorf(__fmul_rn(v.y, inv)), mb1);
        const int i2 = (int)__fsub_rn(floorf(__fmul_rn(v.z, inv)), mb2);
        key = (uint32_t)i0 + (uint32_t)i1 * si.mul1 + (uint32_t)i2 * si.mul2;
      }
      keys[si.off + e] = key;
      count_digits(sh, key);
    }
  }
  __syncthreads();
  flush_digits(sh, totals, n_slots, slot);
}

// A.1 steps 8-9: float centroid per run (voxel), summed in ascending input order — (((p0 + p1) + p2) + ...) exactly as
// PCL's CentroidPoint — and written in ascending key order.  ONE kernel over the sorted (key, index) pairs:
//   * a tile (2048 sorted positions) loads its keys and gathers its points raw[vals[e]] into shared memory — all loads of a
//     thread independent, no sorted copy of the cloud in global memory;
//   * run heads are counted, and the tile's first output rank comes from a decoupled look-back over the earlier tiles of the
//     slot (same status words / tickets as the sort); the last live tile writes n_pts;
//   * the thread that owns a head walks its run through shared memory (continuing in global memory when the run leaves the
//     tile).  Runs longer than kLongRun are only queued: a serial walk needs ~0.4 us per point once it leaves shared memory, and
//     map-sized clouds have voxels with thousands of points;
//   voxel_long_centroid_kernel  one warp per queued run: 32 lanes fetch 32 points at once, then the warp consumes them in
//                               order through shuffles, so the additions stay strictly sequential but never wait for loads.
// Pass-through slots (overflow) are copied here too.
// (Round 1: heads, scan, gather, centroid = four kernels, with the gathered cloud written to and re-read from global memory.)
constexpr uint32_t kLongRun = 64;

__global__ void __launch_bounds__(kSortThreads) voxel_centroid_kernel(SlotInfo* __restrict__ slots, TileMap tm, const uint32_t* __restrict__ slot_tile_begin,
                                                                       const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                                       uint64_t* __restrict__ status, uint32_t* __restrict__ ticket, uint32_t epoch,
                                                                       float4* __restrict__ work, uint4* __restrict__ long_runs, uint32_t* __restrict__ n_long,
                                                                       int32_t* __restrict__ flags) {
  __shared__ float sx[kSortTile], sy[kSortTile], sz[kSortTile];
  __shared__ uint32_t sk[kSortTile];
  __shared__ uint16_t s_head[kSortTile];  // tile positions of the run heads, in order
  __shared__ uint32_t wsum[8];
  __shared__ uint32_t s_tile, s_base;
  if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const uint32_t t = s_tile;
  const uint32_t slot = tm.tile_slot[t], first = tm.tile_first[t];
  SlotInfo& si = slots[slot];
  if (si.overflow) {  // working cloud = raw cloud verbatim
#pragma unroll
    for (int j = 0; j < kSortTile / kSortThreads; ++j) {
      const uint32_t e = first + j * kSortThreads + threadIdx.x;
      if (e < si.n_raw) work[si.off + e] = __ldg(si.raw + e);
    }
    return;
  }
  const uint32_t n = si.n_finite;
  if (first >= n) return;  // dead tiles are a suffix of their slot
  const uint32_t* k = keys + si.off;
  const uint32_t* v = vals + si.off;
  const float4* raw = si.raw;
  const uint32_t live = min(n - first, (uint32_t)kSortTile);
#pragma unroll
  for (int j = 0; j < kSortTile / kSortThreads; ++j) {
    const uint32_t i = j * kSortThreads + threadIdx.x;
    if (i < live) {
      const float4 p = __ldg(raw + v[first + i]);
      sk[i] = k[first + i]; sx[i] = p.x; sy[i] = p.y; sz[i] = p.z;
    }
  }
  __syncthreads();
  constexpr int kPer = kSortTile / kSortThreads;
  const uint32_t i0 = threadIdx.x * kPer;  // kPer consecutive sorted positions per thread
  uint32_t head_mask = 0, cnt = 0;
  uint32_t prev = i0 > 0 ? sk[min(i0, live) - 1] : (first > 0 ? k[first - 1] : 0u);
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const uint32_t i = i0 + j;
    if (i < live) {
      const uint32_t kk = sk[i];
      if (first + i == 0 || kk != prev) { head_mask |= 1u << j; ++cnt; }
      prev = kk;
    }
  }
  // block exclusive scan of cnt
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { uint32_t u = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += u; }
  if (lane == 31) wsum[w] = incl;
  __syncthreads();
  if (w == 0) {  // warp 0 publishes the tile's head count and looks back, 32 earlier tiles per step, for its first rank
    uint32_t total = lane < 8 ? wsum[lane] : 0u;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) total += __shfl_xor_sync(0xFFFFFFFFu, total, o);
    total = __shfl_sync(0xFFFFFFFFu, total, 0);
    const uint64_t tag = uint64_t(epoch) << 32;
    const uint32_t begin = slot_tile_begin[slot];
    uint64_t* mine = status + size_t(t) * 256;
    if (lane == 0) lb_store(mine, tag | (uint64_t(t == begin ? kLbInclusive : kLbAggregate) << 30) | total);
    uint32_t excl = 0;
    if (t != begin) {
      long long q = (long long)t - 1;
      for (;;) {
        const long long qi = q - lane;
        uint64_t x = tag | (uint64_t(kLbInclusive) << 30);  // lanes before the slot's first tile: inclusive, nothing to add
        if (qi >= (long long)begin) {
          const uint64_t* theirs = status + size_t(qi) * 256;
          x = lb_load(theirs);
          uint32_t spin = 0;
          while (uint32_t(x >> 32) != epoch) {
            if (++spin > kLbSpinLimit) { atomicOr(&flags[0], kErrSortStall); x = tag | (uint64_t(kLbInclusive) << 30); break; }
            __nanosleep(20);
            x = lb_load(theirs);
          }
        }
        const uint32_t inclusive = __ballot_sync(0xFFFFFFFFu, (uint32_t(x) >> 30) == kLbInclusive);
        const int stop = inclusive ? __ffs(inclusive) - 1 : 31;  // nearest tile that already knows its prefix
        uint32_t add = lane <= stop ? (uint32_t(x) & kLbValueMask) : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) add += __shfl_xor_sync(0xFFFFFFFFu, add, o);
        excl += add;
        if (inclusive) break;
        q -= 32;
      }
      if (lane == 0) lb_store(mine, tag | (uint64_t(kLbInclusive) << 30) | (excl + total));
    }
    if (lane == 0) {
      s_base = excl;
      if (first + live == n) si.n_pts = excl + total;  // last live tile of the slot: the number of voxels
    }
  }
  __syncthreads();
  // Heads are compacted into a list and dealt out to consecutive threads: with one thread walking the heads of its own 8
  // positions only 3 of 32 lanes were busy in the walk (ncu, profiles/r02_summary.md), and the centroids of a warp now land on
  // consecutive addresses.
  uint32_t lr = incl - cnt, heads = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) { if (i < w) lr += wsum[i]; heads += wsum[i]; }
#pragma unroll
  for (int j = 0; j < kPer; ++j)
    if (head_mask & (1u << j)) s_head[lr++] = (uint16_t)(i0 + j);
  __syncthreads();
  float4* out = work + si.off;
  for (uint32_t h = threadIdx.x; h < heads; h += kSortThreads) {
    const uint32_t i = s_head[h], e = first + i, rank = s_base + h;
    const uint32_t kk = sk[i];
    if (e + kLongRun < n && k[e + kLongRun] == kk) {  // sorted keys: the run has more than kLongRun points
      long_runs[atomicAdd(n_long, 1u)] = make_uint4(slot, e, rank, 0u);
      continue;
    }
    float ax = 0.f, ay = 0.f, az = 0.f;
    uint32_t l = i;
    do {
      ax = __fadd_rn(ax, sx[l]); ay = __fadd_rn(ay, sy[l]); az = __fadd_rn(az, sz[l]);
      ++l;
    } while (l < live && sk[l] == kk);
    uint32_t g = first + l;
    if (l == live) {  // the run may continue in the next tile(s)
      while (g < n && k[g] == kk) {
        const float4 p = __ldg(raw + v[g]);
        ax = __fadd_rn(ax, p.x); ay = __fadd_rn(ay, p.y); az = __fadd_rn(az, p.z);
        ++g;
      }
    }
    const float c = (float)(g - e);
    out[rank] = make_float4(__fdiv_rn(ax, c), __fdiv_rn(ay, c), __fdiv_rn(az, c), 1.0f);
  }
}

// Three lanes of the warp carry the x, y and z sums.  A batch of 32 gathered points is staged in shared memory and every lane
// then reads component (lane & 3) of point j: one LDS + one FADD per point for all three chains, 4 cycles of dependent latency
// per point.  (Fed by shuffles — 3 SHFL + 3 FADD per point, each FADD waiting for its shuffle — the same loop took ~35 cycles per
// point: 358 us on the 5289-point voxels of the 2M-point cloud at 0.2 m, profiles/r02_summary.md.)
__global__ void __launch_bounds__(256, 2) voxel_long_centroid_kernel(const SlotInfo* __restrict__ slots, const uint32_t* __restrict__ keys,
                                                                  const uint32_t* __restrict__ vals, float4* __restrict__ work,
                                                                  const uint4* __restrict__ long_runs, const uint32_t* __restrict__ n_long) {
  const uint32_t FULL = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const uint32_t warps = gridDim.x * (blockDim.x >> 5);
  // One warp walks one run, so its own look-ahead must hide the loads, and a warp issues in order: a point load that waits for
  // its index stalls everything behind it.  Two stages: keys + indices are fetched 2 x kDepth batches ahead, the points kDepth
  // batches ahead with indices that arrived an iteration ago — no load ever waits.  (Index and point fetched in the same
  // iteration cost one L2 round trip per batch: 27 cycles per point instead of ~7.)
  constexpr int kDepth = 8;
  __shared__ float4 s_pts[8][2][32];  // per warp: two staging buffers, so that one __syncwarp per batch is enough
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  const int comp = lane & 3;
  for (uint32_t q = blockIdx.x * (blockDim.x >> 5) + w; q < *n_long; q += warps) {
    const uint4 job = long_runs[q];
    const SlotInfo& si = slots[job.x];
    const uint32_t n = si.n_finite;
    const uint32_t* k = keys + si.off;
    const uint32_t* v = vals + si.off;
    const float4* raw = si.raw;
    const uint32_t kk = k[job.y];
    // The run ends where the key changes (sorted keys: its members are a prefix of every batch).  The keys ride along with the
    // points, so the end is found by the walk itself — a separate gallop + binary search was a chain of ~15 dependent loads.
    float acc = 0.f;
    float4 buf[kDepth];
    uint32_t nk[kDepth], nv[kDepth];
    bool in[kDepth];
#pragma unroll
    for (int d = 0; d < kDepth; ++d) {
      const uint32_t e = job.y + d * 32 + lane, e2 = e + kDepth * 32;
      const uint32_t ke = e < n ? k[e] : ~kk, ve = e < n ? v[e] : 0u;
      nk[d] = e2 < n ? k[e2] : ~kk; nv[d] = e2 < n ? v[e2] : 0u;
      in[d] = ke == kk;
      buf[d] = in[d] ? __ldg(raw + ve) : zero;
    }
    uint32_t len = 0;
    int stage = 0;
    for (uint32_t b = job.y;; b += 32 * kDepth) {
      bool more = true;
#pragma unroll
      for (int d = 0; d < kDepth; ++d) {
        const float4 p = buf[d];
        const int take = __popc(__ballot_sync(FULL, in[d]));
        in[d] = nk[d] == kk;                                         // the batch kDepth ahead: its index is here already
        buf[d] = in[d] ? __ldg(raw + nv[d]) : zero;
        const uint32_t e2 = b + (d + 2 * kDepth) * 32 + lane;      // and the index of the batch 2 x kDepth ahead
        nk[d] = e2 < n ? k[e2] : ~kk; nv[d] = e2 < n ? v[e2] : 0u;
        if (more) {
          s_pts[w][stage][lane] = p;
          __syncwarp();
          const float* f = reinterpret_cast<const float*>(&s_pts[w][stage][0]) + comp;
          if (take == 32) {
#pragma unroll
            for (int j = 0; j < 32; ++j) acc = __fadd_rn(acc, f[4 * j]);
          } else {
            for (int j = 0; j < take; ++j) acc = __fadd_rn(acc, f[4 * j]);
          }
          stage ^= 1;
          len += take;
          if (take < 32) more = false;
        }
      }
      if (!more) break;
    }
    __syncwarp();
    const float sx = __shfl_sync(FULL, acc, 0), sy = __shfl_sync(FULL, acc, 1), sz = __shfl_sync(FULL, acc, 2);
    const float c = (float)len;
    if (lane == 0) work[si.off + job.z] = make_float4(__fdiv_rn(sx, c), __fdiv_rn(sy, c), __fdiv_rn(sz, c), 1.0f);
  }
}

// overflow / pass-through slots: working cloud = raw cloud verbatim
__global__ void __launch_bounds__(kSortThreads) voxel_passthrough_kernel(const SlotInfo* __restrict__ slots, TileMap tm, float4* __restrict__ work) {
  const uint32_t t = blockIdx.x;
  const uint32_t slot = tm.tile_slot[t], first = tm.tile_first[t];
  const SlotInfo& si = slots[slot];
  if (!si.overflow) return;
#pragma unroll
  for (int j = 0; j < kSortTile / kSortThreads; ++j) {
    const uint32_t e = first + j * kSortThreads + threadIdx.x;
    if (e < si.n_raw) work[si.off + e] = si.raw[e];
  }
}

void run_voxel(Workspace& ws, float leaf, uint32_t* leaf_keys) {
  if (ws.n_tiles == 0) {  // all clouds empty: n_pts stays 0
    return;
  }
  cudaStream_t st = ws.stream;
  {  // how much of a raw cloud the last batch with this leaf size kept: sizes the grids of the kernels behind the filter (internal.h)
    static const float pinned = [] { const char* e = getenv("S3D_GRID_FRAC"); return e ? (float)atof(e) : 0.f; }();
    ws.batch_leaf = leaf > 0.f ? leaf : 0.f;
    const auto it = ws.learned_frac.find(ws.batch_leaf);
    ws.grid_frac = pinned > 0.f ? std::min(1.f, pinned) : (leaf > 0.f && it != ws.learned_frac.end() ? it->second : 1.f);
  }
  StageTimer timer(ws, kStageVoxel);
  SlotInfo* slots = ws.slots.as<SlotInfo>();
  TileMap tm{ws.tile_slot.as<uint32_t>(), ws.tile_first.as<uint32_t>(), ws.n_tiles};
  uint32_t* bbox_done = ws.flags.as<uint32_t>() + 10;  // flags are zeroed by setup_batch; the kernel leaves the counter zero
  bbox_kernel<kCountRaw><<<ws.n_tiles, kSortThreads, 0, st>>>(slots, tm, ws.work.as<float4>(), ws.n_slots, bbox_done, VoxelParams{leaf});
  ++ws.launches;
  if (leaf > 0.f) {
    uint32_t* keys[2] = {ws.keys0.as<uint32_t>(), ws.keys1.as<uint32_t>()};
    uint32_t* vals[2] = {ws.vals0.as<uint32_t>(), ws.vals1.as<uint32_t>()};
    if (leaf_keys) S3D_CUDA(cudaMemsetAsync(keys[0], 0xFF, 4 * size_t(ws.total), st));  // skipped / overflow points report 0xFFFFFFFF
    const SortState ss = ws.sort_state();
    sort_clear_aux(st, ss, ws.n_slots);
    voxel_keys_kernel<<<ws.n_tiles, kSortThreads, 0, st>>>(slots, tm, ws.n_slots, keys[0], ss.aux);
    ++ws.launches;
    if (leaf_keys) S3D_CUDA(cudaMemcpyAsync(leaf_keys, keys[0], 4 * size_t(ws.total), cudaMemcpyDeviceToDevice, st));
    radix_sort_segmented(st, slots, ws.n_slots, tm, ws.slot_tile_begin.as<uint32_t>(), keys, vals, ss, kCountRaw, /*digits_done=*/true, &ws.launches);
    uint32_t* n_long = ws.flags.as<uint32_t>() + 8;  // flags[8]: number of queued long runs (flags are zeroed by setup_batch)
    voxel_centroid_kernel<<<ws.n_tiles, kSortThreads, 0, st>>>(slots, tm, ws.slot_tile_begin.as<uint32_t>(), keys[0], vals[0], ss.status, sort_ticket(ss, ws.n_slots, kSortPasses),
                                                               sort_next_epoch(st, ss), ws.work.as<float4>(), ws.long_runs.as<uint4>(), n_long, ss.flags);
    voxel_long_centroid_kernel<<<ws.n_sms * 2, 256, 0, st>>>(slots, keys[0], vals[0], ws.work.as<float4>(), ws.long_runs.as<uint4>(), n_long);
    ws.launches += 2;
  } else {
    voxel_passthrough_kernel<<<ws.n_tiles, kSortThreads, 0, st>>>(slots, tm, ws.work.as<float4>());
    ++ws.launches;
  }
  S3D_CUDA(cudaGetLastError());
}

}  // namespace s3d
