// ransac.cu — PointCloudSensor::fillGroundPlane (slam3d/sensor/pcl/PointCloudSensor.cpp:362-388): pcl::RandomSampleConsensus with
// SampleConsensusModelPlane, then rings of points laid into the plane.  Arithmetic in ransac_math.h; DESIGN.md 6f.
//
// PCL's loop is sequential, but its random samples never depend on the inlier counts.  So one device thread runs the sampler
// ahead (MT19937 state and the shuffled index array stay in device memory between blocks) and emits the next B planes, a
// counting kernel scores all B planes against all points at once, and the host replays the loop's decisions on the B counts in
// loop order.  If the loop has not ended, the next block follows.  Planes sampled after the loop's end are discarded; they do
// not disturb anything the loop saw.
#include <cstdlib>

#include "internal.h"
#include "ransac_math.h"

namespace s3d {

namespace {

constexpr int kScoreThreads = 256;
constexpr int kScorePts = 4;       // points per thread, held in registers for the whole block of planes
constexpr int kTile = 2048;        // points per CTA of the inlier compaction (256 threads x 8 consecutive points)

struct SamplerState {
  uint32_t mt[kMtWords];
  int32_t mti;
  int32_t ended;                   // an empty selection was emitted: every later slot is empty too
  uint32_t pad[2];
};

// shuffled_indices_ = 0..n-1, RNG seeded with 12345u
__global__ void ransac_init_kernel(uint32_t* __restrict__ shuffled, uint32_t n, SamplerState* __restrict__ st) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) shuffled[i] = i;
  if (blockIdx.x == 0 && threadIdx.x == 0) { int32_t mti; mt_seed(st->mt, mti, kRansacSeed); st->mti = mti; st->ended = 0; }
}

// The next `count` iterations of the loop, in order: plane (NaN for flagged slots, so that they count nothing) and
// (sample, flag).  One thread; the MT state lives in shared memory while it runs.
__global__ void __launch_bounds__(32) ransac_sample_kernel(const float4* __restrict__ pts, uint32_t n, uint32_t* __restrict__ shuffled,
                                                           SamplerState* __restrict__ st, int count, float4* __restrict__ planes,
                                                           uint4* __restrict__ sel) {
  __shared__ uint32_t mt[kMtWords];
  for (int i = threadIdx.x; i < kMtWords; i += 32) mt[i] = st->mt[i];
  __syncwarp();
  if (threadIdx.x == 0) {
    int32_t mti = st->mti;
    int32_t ended = st->ended;
    uint32_t s[3] = {shuffled[0], shuffled[1], shuffled[2]};
    const float qnan = __int_as_float(0x7FC00000);
    for (int b = 0; b < count; ++b) {
      float4 plane = make_float4(qnan, qnan, qnan, qnan);
      uint32_t smp[3] = {0, 0, 0};
      int flag = kRansacNoSample;
      if (!ended) {
        flag = ransac_next_hypothesis(mt, mti, shuffled, s, n, pts, &plane, smp);
        if (flag == kRansacNoSample) ended = 1;
        if (flag != kRansacScored) plane = make_float4(qnan, qnan, qnan, qnan);
      }
      planes[b] = plane;
      sel[b] = make_uint4(smp[0], smp[1], smp[2], (uint32_t)flag);
    }
    shuffled[0] = s[0]; shuffled[1] = s[1]; shuffled[2] = s[2];
    st->mti = mti; st->ended = ended;
  }
  __syncwarp();
  for (int i = threadIdx.x; i < kMtWords; i += 32) st->mt[i] = mt[i];
}

// counts[h] += points with distance < t, for the `count` planes of the block.  Each thread keeps kScorePts points in registers
// and tests them against every plane (from shared memory); a warp sums one plane with ballot + popc, a CTA in shared memory and
// the grid with one integer atomic per (CTA, plane): integer sums do not depend on the schedule.
__global__ void __launch_bounds__(kScoreThreads) ransac_score_kernel(const float4* __restrict__ pts, uint32_t n, const float4* __restrict__ planes,
                                                                     int count, float t, uint32_t* __restrict__ counts) {
  extern __shared__ float4 s_planes[];
  uint32_t* s_count = reinterpret_cast<uint32_t*>(s_planes + count);
  for (int h = threadIdx.x; h < count; h += kScoreThreads) { s_planes[h] = planes[h]; s_count[h] = 0; }
  float px[kScorePts], py[kScorePts], pz[kScorePts];
  const uint32_t base = blockIdx.x * (kScoreThreads * kScorePts) + threadIdx.x;
#pragma unroll
  for (int j = 0; j < kScorePts; ++j) {
    const uint32_t i = base + j * kScoreThreads;
    const float4 p = i < n ? pts[i] : make_float4(__int_as_float(0x7FC00000), 0.f, 0.f, 0.f);  // NaN: never an inlier
    px[j] = p.x; py[j] = p.y; pz[j] = p.z;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  for (int h = 0; h < count; ++h) {
    const float4 m = s_planes[h];
    uint32_t c = 0;
#pragma unroll
    for (int j = 0; j < kScorePts; ++j) c += __popc(__ballot_sync(0xFFFFFFFFu, ransac_distance(m, px[j], py[j], pz[j]) < t));
    if (lane == 0 && c) atomicAdd(&s_count[h], c);
  }
  __syncthreads();
  for (int h = threadIdx.x; h < count; h += kScoreThreads)
    if (s_count[h]) atomicAdd(&counts[h], s_count[h]);
}

// selectWithinDistance, order-preserving (the compaction scheme of map.cu): inliers per tile, exclusive scan over the tiles
// (keep_scan_kernel), scatter of the indices
__global__ void __launch_bounds__(256) ransac_inlier_count_kernel(const float4* __restrict__ pts, uint32_t n, float4 m, float t,
                                                                  uint32_t* __restrict__ tile_counts) {
  __shared__ uint32_t wsum[8];
  constexpr int kPer = kTile / 256;
  const uint32_t e0 = blockIdx.x * kTile + threadIdx.x * kPer;
  uint32_t c = 0;
#pragma unroll
  for (int j = 0; j < kPer; ++j)
    if (e0 + j < n) { const float4 p = pts[e0 + j]; c += ransac_distance(m, p.x, p.y, p.z) < t ? 1u : 0u; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) { uint32_t s = 0; for (int i = 0; i < 8; ++i) s += wsum[i]; tile_counts[blockIdx.x] = s; }
}

__global__ void __launch_bounds__(256) ransac_inlier_scatter_kernel(const float4* __restrict__ pts, uint32_t n, float4 m, float t,
                                                                    const uint32_t* __restrict__ tile_offsets, uint32_t* __restrict__ out) {
  __shared__ uint32_t wsum[8];
  constexpr int kPer = kTile / 256;
  const uint32_t e0 = blockIdx.x * kTile + threadIdx.x * kPer;
  uint32_t bits = 0;
#pragma unroll
  for (int j = 0; j < kPer; ++j)
    if (e0 + j < n) { const float4 p = pts[e0 + j]; if (ransac_distance(m, p.x, p.y, p.z) < t) bits |= 1u << j; }
  const uint32_t c = __popc(bits);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t incl = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += u; }
  if (lane == 31) wsum[w] = incl;
  __syncthreads();
  uint32_t pos = tile_offsets[blockIdx.x] + incl - c;
  for (int i = 0; i < w; ++i) pos += wsum[i];
#pragma unroll
  for (int j = 0; j < kPer; ++j) if (bits & (1u << j)) out[pos++] = e0 + j;
}

// point (ring i, angle j) at i * n_angles + j: reference order, ring-major
__global__ void __launch_bounds__(256) ground_fill_kernel(const double* __restrict__ rings, uint32_t n_rings, const double* __restrict__ sin_a,
                                                          const double* __restrict__ cos_a, uint32_t n_angles, double n0, double n1, double n2,
                                                          double offset, float4* __restrict__ out) {
  const uint64_t total = (uint64_t)n_rings * n_angles;
  const double n[3] = {n0, n1, n2};
  for (uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; e < total; e += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t i = (uint32_t)(e / n_angles), j = (uint32_t)(e % n_angles);
    out[e] = ground_fill_point(n, offset, rings[i], sin_a[j], cos_a[j]);
  }
}

int ransac_block_size() {
  static const int b = [] { const char* e = getenv("S3D_RANSAC_BLOCK"); const int v = e ? atoi(e) : 0; return v > 0 ? std::min(v, 2048) : 256; }();
  return b;
}

}  // namespace

RansacFit run_ransac_plane(Workspace& ws, const float4* pts, uint32_t n, double threshold, int max_iterations, double probability,
                           bool want_inliers) {
  RansacFit fit;
  const int B = ransac_block_size();
  const float t = ransac_float_threshold(threshold);
  // device layout of ws.ransac: state | planes[B] | sel[B] | counts[B]; the last three are read back in one copy
  const size_t state_bytes = (sizeof(SamplerState) + 255) & ~size_t(255);
  const size_t blk_bytes = (size_t)B * (16 + 16 + 4);
  ws.ransac.reserve(state_bytes + blk_bytes);
  ws.ransac_idx.reserve(4 * (size_t)n);
  ws.h_ransac.reserve(blk_bytes);
  SamplerState* st = reinterpret_cast<SamplerState*>(ws.ransac.p);
  float4* d_planes = reinterpret_cast<float4*>(ws.ransac.as<char>() + state_bytes);
  uint4* d_sel = reinterpret_cast<uint4*>(d_planes + B);
  uint32_t* d_counts = reinterpret_cast<uint32_t*>(d_sel + B);
  const float4* h_planes = ws.h_ransac.as<float4>();
  const uint4* h_sel = reinterpret_cast<const uint4*>(h_planes + B);
  const uint32_t* h_counts = reinterpret_cast<const uint32_t*>(h_sel + B);
  uint32_t* shuffled = ws.ransac_idx.as<uint32_t>();

  ransac_init_kernel<<<std::min<uint32_t>((n + 255) / 256, 4 * ws.n_sms), 256, 0, ws.stream>>>(shuffled, n, st);
  ++ws.launches;
  RansacReplay R(n, max_iterations, probability);
  const uint32_t score_grid = (n + kScoreThreads * kScorePts - 1) / (kScoreThreads * kScorePts);
  while (R.wants_more()) {
    const int count = (int)std::min<uint64_t>((uint64_t)B, R.remaining_bound());
    ransac_sample_kernel<<<1, 32, 0, ws.stream>>>(pts, n, shuffled, st, count, d_planes, d_sel);
    S3D_CUDA(cudaMemsetAsync(d_counts, 0, 4 * (size_t)count, ws.stream));
    ransac_score_kernel<<<score_grid, kScoreThreads, (size_t)count * 20, ws.stream>>>(pts, n, d_planes, count, t, d_counts);
    ws.launches += 2;
    S3D_CUDA(cudaGetLastError());
    S3D_CUDA(cudaMemcpyAsync(ws.h_ransac.p, d_planes, blk_bytes, cudaMemcpyDeviceToHost, ws.stream));
    ws.sync();
    ws.d2h += blk_bytes;
    for (int b = 0; b < count && R.wants_more(); ++b) {
      const float plane[4] = {h_planes[b].x, h_planes[b].y, h_planes[b].z, h_planes[b].w};
      R.consume((int)h_sel[b].w, h_counts[b], plane);
    }
  }
  fit.iterations = R.iterations;
  fit.ok = R.have_model;
  fit.n_inliers = R.best_count;
  for (int i = 0; i < 4; ++i) fit.coeff[i] = R.best[i];
  if (!fit.ok || !want_inliers) return fit;
  const uint32_t n_tiles = (n + kTile - 1) / kTile;
  ws.map_aux.reserve(4 * ((size_t)n_tiles + 1) + 4 * (size_t)n);
  uint32_t* tile_counts = ws.map_aux.as<uint32_t>();
  uint32_t* d_total = tile_counts + n_tiles;
  uint32_t* d_out = d_total + 1;
  const float4 m = make_float4(fit.coeff[0], fit.coeff[1], fit.coeff[2], fit.coeff[3]);
  ransac_inlier_count_kernel<<<n_tiles, 256, 0, ws.stream>>>(pts, n, m, t, tile_counts);
  keep_scan_kernel<<<1, 32, 0, ws.stream>>>(n_tiles, tile_counts, d_total);
  ransac_inlier_scatter_kernel<<<n_tiles, 256, 0, ws.stream>>>(pts, n, m, t, tile_counts, d_out);
  ws.launches += 3;
  S3D_CUDA(cudaGetLastError());
  uint32_t* h_total = ws.h_small.as<uint32_t>();
  S3D_CUDA(cudaMemcpyAsync(h_total, d_total, 4, cudaMemcpyDeviceToHost, ws.stream));
  ws.sync();
  ws.d2h += 4;
  if (*h_total != fit.n_inliers) throw CudaError{"RANSAC inlier compaction disagrees with the count of the best plane"};
  fit.inliers_dev = d_out;
  return fit;
}

void run_ground_fill(Workspace& ws, const float coeff[4], const std::vector<double>& rings, const std::vector<double>& sin_a,
                     const std::vector<double>& cos_a, float4* dev_out) {
  const uint64_t total = (uint64_t)rings.size() * sin_a.size();
  if (total == 0) return;
  const size_t nr = rings.size(), na = sin_a.size();
  ws.map_aux.reserve(8 * (nr + 2 * na));
  double* d = ws.map_aux.as<double>();
  S3D_CUDA(cudaMemcpyAsync(d, rings.data(), 8 * nr, cudaMemcpyHostToDevice, ws.stream));
  S3D_CUDA(cudaMemcpyAsync(d + nr, sin_a.data(), 8 * na, cudaMemcpyHostToDevice, ws.stream));
  S3D_CUDA(cudaMemcpyAsync(d + nr + na, cos_a.data(), 8 * na, cudaMemcpyHostToDevice, ws.stream));
  ws.h2d += 8 * (nr + 2 * na);
  const uint32_t grid = (uint32_t)std::min<uint64_t>((total + 255) / 256, 8 * (uint64_t)ws.n_sms);
  ground_fill_kernel<<<grid, 256, 0, ws.stream>>>(d, (uint32_t)nr, d + nr, d + nr + na, (uint32_t)na, (double)coeff[0], (double)coeff[1],
                                                  (double)coeff[2], (double)coeff[3], dev_out);
  ++ws.launches;
  S3D_CUDA(cudaGetLastError());
}

}  // namespace s3d
