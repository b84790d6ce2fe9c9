// ndt.cu — the NDT branch of slam3d's align(): pcl::NormalDistributionsTransform as driven by doNDT
// (slam3d/sensor/pcl/PointCloudSensor.cpp:84-117, switch case :145-148).  SURVEY 8f rank 4.
//
// Per registration (pair p: slot 2p = fixed cloud B = PCL target, slot 2p+1 = moving cloud A = PCL source):
//   target grid   VoxelGridCovariance at `resolution` over B's (already voxel-filtered) working cloud: PCL voxel keys ->
//                 the stable segmented radix sort of sort.cuh -> one thread per voxel sums its points in input order
//                 (float centroid, double mean / outer products) -> Gaussian (ndt_math.h) -> leaf array in ascending key
//                 order (= order of PCL's centroid cloud) + an open-addressing hash  voxel key -> leaf.
//   evaluation    ndt_eval_kernel, one thread per moving point: q = final_transformation_ * p (float se3 form), the
//                 kd-tree radius search of PCL (all centroids with d2 < resolution^2, ordered by (d2, index)) becomes a
//                 probe of the 3x3x3 voxels around q's own voxel (a centroid lies in its voxel; the block widens to
//                 5x5x5 when q sits within 1e-3 of a voxel face or some centroid was rounded out of its voxel, so the
//                 result is exact), then score, gradient (6) and Hessian (36) of eq. 6.9/6.12/6.13 in FP64, reduced by
//                 a fixed shuffle tree to one partial per 256-point tile.  NDT_OMP with S3D_NDT_OMP_DIRECT7 launches the
//                 DIRECT7 instantiation instead: pclomp's 7 fixed cells (own voxel + 6 face neighbours) in offset order.
//   control       ndt_ctrl_kernel, one CTA per pair: fixed-order sum of the tile partials, then ONE thread advances
//                 computeTransformation / computeStepLengthMT (resumable state machine, ndt_math.h) to the next
//                 evaluation or to the end.  Pairs of a batch advance independently; the host polls one counter.
//   fitness       getFitnessScore(max_correspondence_distance) on the NN grid of B (nn_search.cuh).
// Bound: latency (27 hash probes + 3-8 leaf loads of 112 B per point, all L2 resident); algorithmic bytes per evaluation
// 16 B per moving point + 112 B per (point, voxel) pair.
#include <cstdio>
#include <cstdlib>

#include "internal.h"
#include "ndt_math.h"
#include "nn_search.cuh"
#include "sort.cuh"

namespace s3d {

// Per-registration state of pair p; its target grid is grids[p] of the launch (built by the raw path, or copied from the
// prepared handle of its fixed cloud).
struct NdtPair {
  float guess[16];
  float T_cur[16];           // final_transformation_: matrix of the pending / last evaluation
  NdtOptState opt;
  NdtAngular ang;            // angular derivative tables at opt.x_t
  double gauss_d1, gauss_d2;
  double fit_range, fit_sum;
  float r2;                  // float(resolution^2)
  uint32_t fit_n;
  int32_t enough;            // both clouds hold >= 100 points (align() :134)
  int32_t active, pending;   // pending: an evaluation at T_cur is requested
};

__device__ __forceinline__ uint32_t ndt_hash_slot(uint32_t key, uint32_t mask) {
  uint32_t h = key * 0x9E3779B1u;
  h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 13;
  return h & mask;
}

// VoxelGridCovariance::applyFilter prologue for B: leaf size, int32 overflow guard, min_b / div_b / divb_mul
__global__ void ndt_params_kernel(const SlotInfo* __restrict__ slots, NdtGridMap map, NdtGrid* __restrict__ grids, uint32_t n_grids) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_grids) return;
  NdtGrid& G = grids[g];
  const SlotInfo& sb = slots[map.slot(g)];
  G.searchable = 0; G.n_voxels = 0; G.n_leaves = 0; G.escaped = 0; G.hash_mask = 0;
  if (sb.n_pts == 0) return;
  if (!(sb.g_max[0] >= sb.g_min[0]) || !(sb.g_max[1] >= sb.g_min[1]) || !(sb.g_max[2] >= sb.g_min[2])) return;  // no finite point
  const float inv = __fdiv_rn(1.0f, G.resolution);
  G.inv_leaf = inv;
  const long long dx = (long long)__fmul_rn(__fsub_rn(sb.g_max[0], sb.g_min[0]), inv) + 1;
  const long long dy = (long long)__fmul_rn(__fsub_rn(sb.g_max[1], sb.g_min[1]), inv) + 1;
  const long long dz = (long long)__fmul_rn(__fsub_rn(sb.g_max[2], sb.g_min[2]), inv) + 1;
  if (dx * dy * dz > 2147483647ll) return;  // "Leaf size is too small for the input dataset": the grid stays empty
  for (int a = 0; a < 3; ++a) {
    G.min_b[a] = (int)floorf(__fmul_rn(sb.g_min[a], inv));
    G.div_b[a] = (int)floorf(__fmul_rn(sb.g_max[a], inv)) - G.min_b[a] + 1;
  }
  G.mul1 = (uint32_t)G.div_b[0];
  G.mul2 = (uint32_t)G.div_b[0] * (uint32_t)G.div_b[1];
  G.searchable = 1;
}

__device__ __forceinline__ uint32_t ndt_voxel_key(const NdtGrid& G, float x, float y, float z) {
  const int i0 = (int)floorf(__fmul_rn(x, G.inv_leaf)) - G.min_b[0];
  const int i1 = (int)floorf(__fmul_rn(y, G.inv_leaf)) - G.min_b[1];
  const int i2 = (int)floorf(__fmul_rn(z, G.inv_leaf)) - G.min_b[2];
  return (uint32_t)i0 + (uint32_t)i1 * G.mul1 + (uint32_t)i2 * G.mul2;
}

// voxel key of every point of a grid slot's working cloud (other slots get key 0: they ride through the segmented sort untouched)
__global__ void __launch_bounds__(kSortThreads) ndt_keys_kernel(const SlotInfo* __restrict__ slots, TileMap tm, const float4* __restrict__ work,
                                                                 NdtGridMap map, const NdtGrid* __restrict__ grids, uint32_t* __restrict__ keys) {
  const uint32_t t = blockIdx.x;
  const uint32_t slot = tm.tile_slot[t], first = tm.tile_first[t];
  const SlotInfo& si = slots[slot];
  if (first >= si.n_pts) return;
  const bool fixed = map.has(slot) && grids[map.grid(slot)].searchable;
#pragma unroll
  for (int j = 0; j < kSortTile / kSortThreads; ++j) {
    const uint32_t e = first + j * kSortThreads + threadIdx.x;
    if (e < si.n_pts) {
      uint32_t key = 0;
      if (fixed) {
        const float4 v = work[si.off + e];
        key = finite3(v.x, v.y, v.z) ? ndt_voxel_key(grids[map.grid(slot)], v.x, v.y, v.z) : kInvalidKey;
      }
      keys[si.off + e] = key;
    }
  }
}

// run starts (voxels) per tile of a grid slot's sorted keys
__global__ void __launch_bounds__(kSortThreads) ndt_heads_kernel(const SlotInfo* __restrict__ slots, TileMap tm, NdtGridMap map,
                                                                  const NdtGrid* __restrict__ grids, const uint32_t* __restrict__ keys,
                                                                  uint32_t* __restrict__ tile_heads) {
  __shared__ uint32_t wsum[8];
  const uint32_t t = blockIdx.x;
  const uint32_t slot = tm.tile_slot[t], first = tm.tile_first[t];
  if (!map.has(slot)) return;
  const SlotInfo& si = slots[slot];
  if (!grids[map.grid(slot)].searchable || first >= si.n_pts) return;
  const uint32_t n = si.n_pts;
  const uint32_t* k = keys + si.off;
  uint32_t c = 0;
#pragma unroll
  for (int j = 0; j < kSortTile / kSortThreads; ++j) {
    const uint32_t e = first + j * kSortThreads + threadIdx.x;
    if (e < n) { const uint32_t kk = k[e]; c += (kk != kInvalidKey && (e == 0 || kk != k[e - 1])) ? 1u : 0u; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) { uint32_t s = 0; for (int i = 0; i < 8; ++i) s += wsum[i]; tile_heads[t] = s; }
}

// one warp per grid: exclusive scan of the tile counts of its slot, number of voxels, hash capacity
__global__ void ndt_scan_kernel(const SlotInfo* __restrict__ slots, NdtGridMap map, NdtGrid* __restrict__ grids,
                                const uint32_t* __restrict__ slot_tile_begin, uint32_t* __restrict__ tile_heads) {
  const uint32_t g = blockIdx.x;
  NdtGrid& G = grids[g];
  if (!G.searchable) return;
  const uint32_t slot = map.slot(g);
  const SlotInfo& si = slots[slot];
  const uint32_t ntiles = (si.n_pts + kSortTile - 1) / kSortTile;
  uint32_t* h = tile_heads + slot_tile_begin[slot];
  const int lane = threadIdx.x;
  uint32_t running = 0;
  for (uint32_t b = 0; b < ntiles; b += 32) {
    const uint32_t t = b + lane;
    const uint32_t v = t < ntiles ? h[t] : 0u;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += u; }
    if (t < ntiles) h[t] = running + incl - v;
    running += __shfl_sync(0xFFFFFFFFu, incl, 31);
  }
  if (lane == 0) {
    G.n_voxels = running;
    uint32_t cap = 4;
    while (cap < 2u * running + 2u) cap <<= 1;
    G.hash_mask = cap - 1u;
  }
}

__global__ void ndt_hash_clear_kernel(const NdtGrid* __restrict__ grids) {
  const NdtGrid& G = grids[blockIdx.y];
  if (!G.searchable) return;
  uint2* tab = G.table;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i <= G.hash_mask; i += gridDim.x * blockDim.x) tab[i] = make_uint2(0xFFFFFFFFu, 0u);
}

// One thread per voxel (run of equal sorted keys): sums in ascending input order (the sort is stable), Gaussian, leaf record,
// hash insertion.  Leaves with fewer than 6 points are recorded with key = kInvalidKey and stay out of the hash; leaves PCL marks
// invalid go into the hash with kNdtLeafInvalid in their key.
__global__ void __launch_bounds__(kSortThreads) ndt_leaf_kernel(const SlotInfo* __restrict__ slots, TileMap tm, NdtGridMap map,
                                                                 NdtGrid* __restrict__ grids, const uint32_t* __restrict__ keys,
                                                                 const uint32_t* __restrict__ vals, const float4* __restrict__ work,
                                                                 const uint32_t* __restrict__ tile_heads) {
  __shared__ uint32_t wsum[8];
  const uint32_t t = blockIdx.x;
  const uint32_t slot = tm.tile_slot[t], first = tm.tile_first[t];
  if (!map.has(slot)) return;
  const SlotInfo& si = slots[slot];
  NdtGrid& G = grids[map.grid(slot)];
  const uint32_t n = si.n_pts;
  if (!G.searchable || first >= n) return;
  const uint32_t* k = keys + si.off;
  const uint32_t* v = vals + si.off;
  const float4* pts = work + si.off;
  constexpr int kPer = kSortTile / kSortThreads;
  const uint32_t e0 = first + threadIdx.x * kPer;
  uint32_t head_mask = 0, cnt = 0;
  uint32_t prev = (e0 > 0 && e0 < n) ? k[e0 - 1] : 0u;
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const uint32_t e = e0 + j;
    if (e < n) {
      const uint32_t kk = k[e];
      if (kk != kInvalidKey && (e == 0 || kk != prev)) { head_mask |= 1u << j; ++cnt; }
      prev = kk;
    }
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += u; }
  if (lane == 31) wsum[w] = incl;
  __syncthreads();
  uint32_t rank = tile_heads[t] + incl - cnt;
  for (int i = 0; i < w; ++i) rank += wsum[i];
  uint2* tab = G.table;
  NdtLeaf* out = G.leaves;
#pragma unroll 1
  for (int j = 0; j < kPer; ++j) {
    if (!(head_mask & (1u << j))) continue;
    const uint32_t e = e0 + j;
    const uint32_t kk = k[e];
    float cs0 = 0.f, cs1 = 0.f, cs2 = 0.f;
    double ms[3] = {0, 0, 0}, cv[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    uint32_t l = e;
    do {
      const float4 pt = pts[v[l]];
      cs0 = __fadd_rn(cs0, pt.x); cs1 = __fadd_rn(cs1, pt.y); cs2 = __fadd_rn(cs2, pt.z);   // leaf.centroid += xyz (float)
      const double d[3] = {(double)pt.x, (double)pt.y, (double)pt.z};
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        ms[a] += d[a];                                                                        // leaf.mean_ += pt3d
#pragma unroll
        for (int b = 0; b < 3; ++b) cv[a][b] += d[a] * d[b];                                  // leaf.cov_ += pt3d pt3d^T
      }
      ++l;
    } while (l < n && k[l] == kk);
    const int nr = (int)(l - e);
    NdtLeaf L;
    L.key = kInvalidKey; L.cx = L.cy = L.cz = 0.f;
    for (int a = 0; a < 3; ++a) L.mean[a] = 0.0;
    for (int a = 0; a < 9; ++a) L.icov[a] = 0.0;
    if (nr >= 6) {  // min_points_per_voxel_
      const float fn = (float)nr;
      L.cx = __fdiv_rn(cs0, fn); L.cy = __fdiv_rn(cs1, fn); L.cz = __fdiv_rn(cs2, fn);
      const bool valid = ndt_finalize_leaf(nr, ms, cv, L.mean, L.icov) && ndt_icov_usable(L.icov);
      L.key = valid ? kk : (kk | kNdtLeafInvalid);
      if (ndt_voxel_key(G, L.cx, L.cy, L.cz) != kk) atomicOr(&G.escaped, 1u);
      atomicAdd(&G.n_leaves, 1u);
      uint32_t s = ndt_hash_slot(kk, G.hash_mask);
      for (;;) {
        if (atomicCAS(&tab[s].x, 0xFFFFFFFFu, kk) == 0xFFFFFFFFu) { tab[s].y = rank; break; }
        s = (s + 1) & G.hash_mask;
      }
    }
    out[rank] = L;
    ++rank;
  }
}

// Registration::align set-up after the grid is known: the <100 gate, and "Voxel grid is not searchable" ends the registration at once
__global__ void ndt_prepare_kernel(const SlotInfo* __restrict__ slots, NdtPair* __restrict__ pairs, const NdtGrid* __restrict__ grids,
                                   uint32_t n_pairs, int32_t* __restrict__ flags) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pairs) return;
  NdtPair& np = pairs[p];
  np.enough = (slots[2 * p + 1].n_pts >= 100 && slots[2 * p].n_pts >= 100) ? 1 : 0;
  if (np.enough && grids[p].searchable && grids[p].n_leaves > 0) {
    np.active = 1; np.pending = 1;  // first computeDerivatives at `transform` with output = guess * input (T_cur = guess)
    ndt_angle_derivatives(np.opt.x_t, np.ang);
    atomicAdd(&flags[1], 1);
  } else {
    np.active = 0; np.pending = 0;
    np.opt.phase = 3; np.opt.converged = 0;
    for (int i = 0; i < 16; ++i) np.T_cur[i] = (i % 5 == 0) ? 1.f : 0.f;  // final_transformation_ keeps align()'s identity
  }
}

constexpr int kNdtMaxCand = 32;

// rank of the leaf under `key`, or kNoIndex (DIRECT7 lookups)
__device__ __forceinline__ uint32_t ndt_hash_find(const uint2* __restrict__ tab, uint32_t mask, uint32_t key) {
  uint32_t s = ndt_hash_slot(key, mask);
  for (;;) {
    const uint2 en = __ldg(tab + s);
    if (en.x == key) return en.y;
    if (en.x == 0xFFFFFFFFu) return kNoIndex;
    s = (s + 1) & mask;
  }
}

// computeDerivatives: one thread per moving point.  kDirect7 = false: PCL's kd-tree radius search (NDT, and NDT_OMP with
// S3D_NDT_OMP_KDTREE).  kDirect7 = true: pclomp's DIRECT7 neighbourhood (NDT_OMP with S3D_NDT_OMP_DIRECT7): the query's own voxel
// and its 6 face neighbours in pclomp's order, cell by float division, leaves with >= 6 points that PCL did not mark invalid.
template <bool kDirect7>
__global__ void __launch_bounds__(kIterTile) ndt_eval_kernel(const SlotInfo* __restrict__ slots, const NdtPair* __restrict__ pairs,
                                                             const NdtGrid* __restrict__ grids, double* __restrict__ part) {
  __shared__ NdtAngular ang;
  __shared__ double wpart[kIterTile / 32][kNdtSums];
  const uint32_t p = blockIdx.y;
  const NdtPair& np = pairs[p];
  if (!np.pending) return;
  const NdtGrid& G = grids[p];
  const SlotInfo& sa = slots[2 * p + 1];
  const uint32_t first = blockIdx.x * kIterTile;
  if (first >= sa.n_pts) return;
  for (int i = threadIdx.x; i < (int)(sizeof(NdtAngular) / sizeof(double)); i += kIterTile)
    reinterpret_cast<double*>(&ang)[i] = reinterpret_cast<const double*>(&np.ang)[i];
  __syncthreads();
  double acc[kNdtSums];
#pragma unroll
  for (int i = 0; i < kNdtSums; ++i) acc[i] = 0.0;
  const uint32_t r = first + threadIdx.x;
  if constexpr (kDirect7) {
    if (r < sa.n_pts) {
      const float4 pt = sa.gpts[r];
      const float3 q = transform_se3(np.T_cur, pt.x, pt.y, pt.z);
      long long ijk[3];
      if (ndt_direct7_cell(q.x, q.y, q.z, G.resolution, ijk)) {
        const uint2* tab = G.table;
        const NdtLeaf* lv = G.leaves;
        uint32_t cr[7];
        int nc = 0;
#pragma unroll
        for (int i = 0; i < 7; ++i) {
          uint32_t key;
          if (!ndt_direct7_key(ijk, i, G.min_b, G.div_b, G.mul1, G.mul2, key)) continue;
          const uint32_t rank = ndt_hash_find(tab, G.hash_mask, key);
          if (rank == kNoIndex) continue;  // no leaf, or fewer than 6 points (those stay out of the hash)
          if (__ldg(&lv[rank].key) & kNdtLeafInvalid) continue;
          cr[nc++] = rank;
        }
        if (nc) {
          const double xo[3] = {(double)pt.x, (double)pt.y, (double)pt.z};
          NdtPointDerivs P;
          ndt_point_derivatives(ang, xo, P);
          for (int i = 0; i < nc; ++i) {
            const double* lp = reinterpret_cast<const double*>(lv + cr[i]);  // [2..4] mean, [5..13] icov
            double ci[9];
            const double xt[3] = {(double)q.x - __ldg(lp + 2), (double)q.y - __ldg(lp + 3), (double)q.z - __ldg(lp + 4)};
#pragma unroll
            for (int a = 0; a < 9; ++a) ci[a] = __ldg(lp + 5 + a);
            ndt_accumulate(P, np.gauss_d1, np.gauss_d2, xt, ci, acc);
            acc[43] += 1.0;
          }
        }
      }
    }
  } else if (r < sa.n_pts) {
    const float4 pt = sa.gpts[r];
    const float3 q = transform_se3(np.T_cur, pt.x, pt.y, pt.z);
    if (finite3(q.x, q.y, q.z)) {
      const float inv = G.inv_leaf;
      const float ux = __fmul_rn(q.x, inv), uy = __fmul_rn(q.y, inv), uz = __fmul_rn(q.z, inv);
      const float fx = floorf(ux), fy = floorf(uy), fz = floorf(uz);
      if (fabsf(fx) < 1.0e9f && fabsf(fy) < 1.0e9f && fabsf(fz) < 1.0e9f) {
        const int cx = (int)fx - G.min_b[0], cy = (int)fy - G.min_b[1], cz = (int)fz - G.min_b[2];
        // a centroid within `resolution` of q lies in the 3x3x3 block around q's voxel unless q sits on a face or the
        // float centroid was rounded out of its voxel: then the block widens on that side
        const bool esc = G.escaped != 0;
        const float ax = ux - fx, ay = uy - fy, az = uz - fz;
        const int lox = (esc || ax < 1e-3f) ? -2 : -1, hix = (esc || ax > 0.999f) ? 2 : 1;
        const int loy = (esc || ay < 1e-3f) ? -2 : -1, hiy = (esc || ay > 0.999f) ? 2 : 1;
        const int loz = (esc || az < 1e-3f) ? -2 : -1, hiz = (esc || az > 0.999f) ? 2 : 1;
        const uint2* tab = G.table;
        const NdtLeaf* lv = G.leaves;
        const uint32_t mask = G.hash_mask;
        float cd[kNdtMaxCand];
        uint32_t ck[kNdtMaxCand], cr[kNdtMaxCand];
        int nc = 0;
        for (int dz = loz; dz <= hiz; ++dz) {
          const int iz = cz + dz;
          if ((unsigned)iz >= (unsigned)G.div_b[2]) continue;
          for (int dy = loy; dy <= hiy; ++dy) {
            const int iy = cy + dy;
            if ((unsigned)iy >= (unsigned)G.div_b[1]) continue;
            for (int dx = lox; dx <= hix; ++dx) {
              const int ix = cx + dx;
              if ((unsigned)ix >= (unsigned)G.div_b[0]) continue;
              const uint32_t key = (uint32_t)ix + (uint32_t)iy * G.mul1 + (uint32_t)iz * G.mul2;
              uint32_t s = ndt_hash_slot(key, mask), rank = kNoIndex;
              for (;;) {
                const uint2 en = __ldg(tab + s);
                if (en.x == key) { rank = en.y; break; }
                if (en.x == 0xFFFFFFFFu) break;
                s = (s + 1) & mask;
              }
              if (rank == kNoIndex) continue;
              const float4 c = __ldg(reinterpret_cast<const float4*>(lv + rank));
              const float d2 = dist2_pcl(q.x, q.y, q.z, c.x, c.y, c.z);
              if (d2 < np.r2 && nc < kNdtMaxCand) {  // FLANN radius search: dist < radius^2, results ordered by (dist, index)
                int i = nc++;
                while (i > 0 && (cd[i - 1] > d2 || (cd[i - 1] == d2 && ck[i - 1] > key))) { cd[i] = cd[i - 1]; ck[i] = ck[i - 1]; cr[i] = cr[i - 1]; --i; }
                cd[i] = d2; ck[i] = key; cr[i] = rank;
              }
            }
          }
        }
        if (nc) {
          const double xo[3] = {(double)pt.x, (double)pt.y, (double)pt.z};
          NdtPointDerivs P;
          ndt_point_derivatives(ang, xo, P);
          for (int i = 0; i < nc; ++i) {
            const double* lp = reinterpret_cast<const double*>(lv + cr[i]);  // [2..4] mean, [5..13] icov
            double ci[9];
            const double xt[3] = {(double)q.x - __ldg(lp + 2), (double)q.y - __ldg(lp + 3), (double)q.z - __ldg(lp + 4)};
#pragma unroll
            for (int a = 0; a < 9; ++a) ci[a] = __ldg(lp + 5 + a);
            ndt_accumulate(P, np.gauss_d1, np.gauss_d2, xt, ci, acc);
            acc[43] += 1.0;
          }
        }
      }
    }
  }
  // fixed reduction tree: butterfly inside each warp, then the 8 warps in order
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < kNdtSums; ++i) {
    double v = acc[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    if (lane == 0) wpart[w][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < kNdtSums) {
    double s = wpart[0][threadIdx.x];
#pragma unroll
    for (int i = 1; i < kIterTile / 32; ++i) s += wpart[i][threadIdx.x];
    part[((size_t)p * gridDim.x + blockIdx.x) * kNdtSums + threadIdx.x] = s;
  }
}

constexpr int kNdtCtrlSubs = 4;

// one CTA per pair: ordered sum of the tile partials, then the optimiser advances to its next evaluation or finishes
__global__ void __launch_bounds__(kNdtCtrlSubs * kNdtSums) ndt_ctrl_kernel(const SlotInfo* __restrict__ slots, NdtPair* __restrict__ pairs,
                                                                            const double* __restrict__ part, uint32_t tiles_per_pair,
                                                                            int32_t* __restrict__ flags) {
  __shared__ double sub[kNdtCtrlSubs][kNdtSums];
  __shared__ double sums[kNdtSums];
  const uint32_t p = blockIdx.x;
  NdtPair& np = pairs[p];
  if (!np.pending) return;
  const uint32_t n_tiles = (slots[2 * p + 1].n_pts + kIterTile - 1) / kIterTile;
  {
    const int m = threadIdx.x % kNdtSums, sb = threadIdx.x / kNdtSums;
    const uint32_t per = (n_tiles + kNdtCtrlSubs - 1) / kNdtCtrlSubs;
    const uint32_t lo = sb * per, hi = min(n_tiles, lo + per);
    const double* src = part + (size_t)p * tiles_per_pair * kNdtSums + m;
    double s = 0.0;
#pragma unroll 4
    for (uint32_t t = lo; t < hi; ++t) s += src[(size_t)t * kNdtSums];
    sub[sb][m] = s;
  }
  __syncthreads();
  if (threadIdx.x < kNdtSums) {
    double s = sub[0][threadIdx.x];
    for (int i = 1; i < kNdtCtrlSubs; ++i) s += sub[i][threadIdx.x];
    sums[threadIdx.x] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (ndt_opt_on_eval(np.opt, sums)) {
      ndt_convert_transform(np.opt.x_t, np.T_cur);  // convertTransform(x_t, final_transformation_)
      ndt_angle_derivatives(np.opt.x_t, np.ang);
    } else {
      np.pending = 0; np.active = 0;
      atomicSub(&flags[1], 1);
    }
  }
}

// getFitnessScore(max_range): transformPointCloud(input, final), 1-NN in B, d2 <= max_range (sic), mean of d2
__global__ void __launch_bounds__(kIterTile) ndt_fitness_kernel(const SlotInfo* __restrict__ slots, const NdtPair* __restrict__ pairs,
                                                                double* __restrict__ fit_partial) {
  __shared__ double ssum[kIterTile];
  __shared__ uint32_t scnt[kIterTile];
  const uint32_t p = blockIdx.y;
  const NdtPair& np = pairs[p];
  if (!np.enough) return;
  const SlotInfo& sb = slots[2 * p];
  const SlotInfo& sa = slots[2 * p + 1];
  const uint32_t first = blockIdx.x * kIterTile;
  if (first >= sa.n_pts) return;
  const uint32_t r = first + threadIdx.x;
  double s = 0.0; uint32_t c = 0;
  if (r < sa.n_pts) {
    const GridView g = make_grid_view(sb);
    const float4 v = sa.gpts[r];
    const float3 q = transform_se3(np.T_cur, v.x, v.y, v.z);
    const NNResult nn = nn_search(g, q.x, q.y, q.z, __double2float_ru(np.fit_range), kNoIndex);
    if (nn.pos != kNoIndex && (double)nn.d2 <= np.fit_range) { s = (double)nn.d2; c = 1; }
  }
  ssum[threadIdx.x] = s; scnt[threadIdx.x] = c;
  __syncthreads();
  for (int o = kIterTile / 2; o > 0; o >>= 1) {  // fixed tree
    if (threadIdx.x < o) { ssum[threadIdx.x] += ssum[threadIdx.x + o]; scnt[threadIdx.x] += scnt[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const size_t tile = (size_t)p * gridDim.x + blockIdx.x;
    fit_partial[2 * tile] = ssum[0];
    fit_partial[2 * tile + 1] = (double)scnt[0];
  }
}

__global__ void ndt_fitness_reduce_kernel(const SlotInfo* __restrict__ slots, NdtPair* __restrict__ pairs, const double* __restrict__ fit_partial,
                                          uint32_t tiles_per_pair, uint32_t n_pairs) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pairs) return;
  NdtPair& np = pairs[p];
  np.fit_sum = 0.0; np.fit_n = 0;
  if (!np.enough) return;
  const uint32_t n_tiles = (slots[2 * p + 1].n_pts + kIterTile - 1) / kIterTile;
  double s = 0.0, c = 0.0;
  for (uint32_t t = 0; t < n_tiles; ++t) { s += fit_partial[2 * ((size_t)p * tiles_per_pair + t)]; c += fit_partial[2 * ((size_t)p * tiles_per_pair + t) + 1]; }
  np.fit_sum = s; np.fit_n = (uint32_t)c;
}

// ------------------------------------------------------------------------------------------------------------------
static void iso_inverse_d(const double T[16], double out[16]) {
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) out[c * 4 + r] = T[r * 4 + c];
  for (int r = 0; r < 3; ++r) { double s = 0; for (int c = 0; c < 3; ++c) s += out[c * 4 + r] * T[12 + c]; out[12 + r] = -s; }
  out[3] = out[7] = out[11] = 0; out[15] = 1;
}
static void m4d_mul_d(const double A[16], const double B[16], double C[16]) {
  for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) { double s = 0; for (int k = 0; k < 4; ++k) s += A[k * 4 + r] * B[c * 4 + k]; C[c * 4 + r] = s; }
}
double rotation_angle_of(const double T[16]);  // gicp.cu: Eigen::AngleAxisd(R).angle()

// VoxelGridCovariance of the slots `map` selects (voxel filter and NN grid must be ready): grid g at resolution[g] lands in
// ws.ndt_grids[g], its leaves and hash table in the workspace's NDT arenas.  Nothing is synchronised.
void run_ndt_grids(Workspace& ws, NdtGridMap map, uint32_t n_grids, const float* resolution) {
  cudaStream_t st = ws.stream;
  ws.ndt_grids.reserve(sizeof(NdtGrid) * std::max<uint32_t>(n_grids, 1));
  ws.h_grids.reserve(sizeof(NdtGrid) * std::max<uint32_t>(n_grids, 1));
  NdtGrid* hg = ws.h_grids.as<NdtGrid>();
  std::vector<size_t> leaf_off(n_grids), hash_off(n_grids);
  size_t leaf_total = 0, hash_total = 0;
  for (uint32_t g = 0; g < n_grids; ++g) {
    const size_t nb = ws.h_n[map.slot(g)];  // raw size of the cloud bounds its voxel count
    leaf_off[g] = leaf_total;
    hash_off[g] = hash_total;
    leaf_total += nb;
    size_t cap = 4;
    while (cap < 2 * nb + 2) cap <<= 1;
    hash_total += cap;
  }
  ws.ndt_leaves.reserve(sizeof(NdtLeaf) * std::max<size_t>(leaf_total, 1));
  ws.ndt_hash.reserve(sizeof(uint2) * std::max<size_t>(hash_total, 4));
  for (uint32_t g = 0; g < n_grids; ++g) {
    memset(&hg[g], 0, sizeof(NdtGrid));
    hg[g].resolution = resolution[g];
    hg[g].leaves = ws.ndt_leaves.as<NdtLeaf>() + leaf_off[g];
    hg[g].table = ws.ndt_hash.as<uint2>() + hash_off[g];
  }
  S3D_CUDA(cudaMemcpyAsync(ws.ndt_grids.p, hg, sizeof(NdtGrid) * n_grids, cudaMemcpyHostToDevice, st));
  const SlotInfo* slots = ws.slots.as<SlotInfo>();
  NdtGrid* grids = ws.ndt_grids.as<NdtGrid>();
  TileMap tm{ws.tile_slot.as<uint32_t>(), ws.tile_first.as<uint32_t>(), ws.n_tiles};
  StageTimer timer(ws, kStageKnn);  // the target's Gaussian voxel grid takes the place of GICP's covariance stage
  uint32_t* keys[2] = {ws.keys0.as<uint32_t>(), ws.keys1.as<uint32_t>()};
  uint32_t* vals[2] = {ws.vals0.as<uint32_t>(), ws.vals1.as<uint32_t>()};
  ndt_params_kernel<<<(n_grids + 63) / 64, 64, 0, st>>>(slots, map, grids, n_grids);
  ndt_keys_kernel<<<ws.n_tiles, kSortThreads, 0, st>>>(slots, tm, ws.work.as<float4>(), map, grids, keys[0]);
  ws.launches += 2;
  radix_sort_segmented(st, slots, ws.n_slots, tm, ws.slot_tile_begin.as<uint32_t>(), keys, vals, ws.sort_state(), kCountPts, /*digits_done=*/false,
                       &ws.launches);
  ndt_heads_kernel<<<ws.n_tiles, kSortThreads, 0, st>>>(slots, tm, map, grids, keys[0], ws.tile_heads.as<uint32_t>());
  ndt_scan_kernel<<<n_grids, 32, 0, st>>>(slots, map, grids, ws.slot_tile_begin.as<uint32_t>(), ws.tile_heads.as<uint32_t>());
  ndt_hash_clear_kernel<<<dim3(32, n_grids), 256, 0, st>>>(grids);
  ndt_leaf_kernel<<<ws.n_tiles, kSortThreads, 0, st>>>(slots, tm, map, grids, keys[0], vals[0], ws.work.as<float4>(), ws.tile_heads.as<uint32_t>());
  ws.launches += 4;
}

// The optimiser of doNDT for every pair of ws's batch; ws.ndt_grids[p] holds the grid of pair p on the device (built by
// run_ndt_grids on this stream, or uploaded from prepared handles).  Fills `out` with the decisions of doNDT (:107-110) and
// align() (:134-135, :167-172).  direct7: every evaluation uses pclomp's DIRECT7 neighbourhood instead of the radius search.
static void ndt_optimise(Workspace& ws, const std::vector<s3d_registration_parameters>& params, const double* guesses, bool direct7,
                         s3d_result* out) {
  const uint32_t np = ws.n_pairs;
  cudaStream_t st = ws.stream;
  const uint32_t tiles_per_pair = std::max<uint32_t>(1, (ws.max_na + kIterTile - 1) / kIterTile);
  ws.ndt_pairs.reserve(sizeof(NdtPair) * np);
  ws.h_pairs.reserve(sizeof(NdtPair) * np);
  NdtPair* hp = ws.h_pairs.as<NdtPair>();
  int max_iter = 0;
  for (uint32_t p = 0; p < np; ++p) {
    const s3d_registration_parameters& cfg = params[p];
    NdtPair& q = hp[p];
    memset(&q, 0, sizeof q);
    for (int i = 0; i < 16; ++i) {
      q.guess[i] = (float)guesses[16 * p + i];  // guess.matrix().cast<float>()  :101
      q.T_cur[i] = q.guess[i];
    }
    double x0[6];
    ndt_initial_state(q.guess, x0);
    ndt_opt_begin(q.opt, x0, cfg.step_size, cfg.transformation_epsilon, cfg.maximum_iterations);
    ndt_gauss_constants((double)cfg.resolution, cfg.outlier_ratio, q.gauss_d1, q.gauss_d2);
    q.fit_range = cfg.max_correspondence_distance;
    q.r2 = (float)((double)cfg.resolution * (double)cfg.resolution);
    max_iter = std::max(max_iter, cfg.maximum_iterations);
  }
  ws.ndt_part.reserve(sizeof(double) * kNdtSums * size_t(tiles_per_pair) * np);
  ws.fit_partial.reserve(sizeof(double) * 2 * size_t(tiles_per_pair) * np);
  S3D_CUDA(cudaMemcpyAsync(ws.ndt_pairs.p, hp, sizeof(NdtPair) * np, cudaMemcpyHostToDevice, st));
  const SlotInfo* slots = ws.slots.as<SlotInfo>();
  NdtPair* pairs = ws.ndt_pairs.as<NdtPair>();
  const NdtGrid* grids = ws.ndt_grids.as<NdtGrid>();
  int32_t* flags = ws.flags.as<int32_t>();
  int32_t* h_flags = ws.h_small.as<int32_t>();
  {
    StageTimer timer(ws, kStageSolve);
    ndt_prepare_kernel<<<(np + 63) / 64, 64, 0, st>>>(slots, pairs, grids, np, flags);
    ++ws.launches;
  }
  const bool trace = getenv("S3D_TRACE") != nullptr;
  dim3 grid(tiles_per_pair, np);
  // every outer iteration needs at least one evaluation, a line search at most 11; 4 evaluate/advance passes per host poll
  const long max_rounds = ((long)std::max(max_iter, 1) * 11 + 2) / 4 + 2;
  for (long round = 0; round < max_rounds; ++round) {
    for (int e = 0; e < 4; ++e) {
      {
        StageTimer timer(ws, kStageIter);
        if (direct7) ndt_eval_kernel<true><<<grid, kIterTile, 0, st>>>(slots, pairs, grids, ws.ndt_part.as<double>());
        else ndt_eval_kernel<false><<<grid, kIterTile, 0, st>>>(slots, pairs, grids, ws.ndt_part.as<double>());
        ++ws.launches;
      }
      {
        StageTimer timer(ws, kStageSolve);
        ndt_ctrl_kernel<<<np, kNdtCtrlSubs * kNdtSums, 0, st>>>(slots, pairs, ws.ndt_part.as<double>(), tiles_per_pair, flags);
        ++ws.launches;
      }
    }
    S3D_CUDA(cudaMemcpyAsync(h_flags, flags, 16, cudaMemcpyDeviceToHost, st));
    ws.sync();
    ws.d2h += 16;
    if (trace && np <= 4) {
      ws.h_grids.reserve(sizeof(NdtGrid) * np);
      NdtGrid* hg = ws.h_grids.as<NdtGrid>();
      S3D_CUDA(cudaMemcpy(hp, pairs, sizeof(NdtPair) * np, cudaMemcpyDeviceToHost));
      S3D_CUDA(cudaMemcpy(hg, grids, sizeof(NdtGrid) * np, cudaMemcpyDeviceToHost));
      for (uint32_t p = 0; p < np; ++p)
        fprintf(stderr, "[s3d ndt] round=%ld pair=%u phase=%d outer=%d line=%d score=%.12g x=(%.9g %.9g %.9g %.9g %.9g %.9g) pairs=%u leaves=%u/%u esc=%u\n", round, p,
                hp[p].opt.phase, hp[p].opt.nr_iterations, hp[p].opt.line_iterations, hp[p].opt.score, hp[p].opt.x[0], hp[p].opt.x[1], hp[p].opt.x[2],
                hp[p].opt.x[3], hp[p].opt.x[4], hp[p].opt.x[5], hp[p].opt.n_pairs_last, hg[p].n_leaves, hg[p].n_voxels, hg[p].escaped);
    }
    if (h_flags[1] <= 0) break;
  }
  {
    StageTimer timer(ws, kStageFitness);
    ndt_fitness_kernel<<<grid, kIterTile, 0, st>>>(slots, pairs, ws.fit_partial.as<double>());
    ndt_fitness_reduce_kernel<<<(np + 63) / 64, 64, 0, st>>>(slots, pairs, ws.fit_partial.as<double>(), tiles_per_pair, np);
    ws.launches += 2;
  }
  S3D_CUDA(cudaMemcpyAsync(hp, pairs, sizeof(NdtPair) * np, cudaMemcpyDeviceToHost, st));
  SlotInfo* hs = ws.h_slots.as<SlotInfo>();
  S3D_CUDA(cudaMemcpyAsync(hs, slots, sizeof(SlotInfo) * ws.n_slots, cudaMemcpyDeviceToHost, st));
  S3D_CUDA(cudaMemcpyAsync(h_flags, flags, 16, cudaMemcpyDeviceToHost, st));
  ws.sync();
  ws.d2h += sizeof(NdtPair) * np + sizeof(SlotInfo) * ws.n_slots + 16;
  ws.collect_spans();
  check_arena(ws, h_flags);
  for (uint32_t p = 0; p < np; ++p) {
    const s3d_registration_parameters& cfg = params[p];
    const NdtPair& q = hp[p];
    s3d_result& r = out[p];
    memset(&r, 0, sizeof r);
    for (int i = 0; i < 16; ++i) r.T[i] = (i % 5 == 0) ? 1.0 : 0.0;
    r.n_source = hs[2 * p].n_pts; r.n_target = hs[2 * p + 1].n_pts;
    if (r.n_target < 100 || r.n_source < 100) { r.status = S3D_TOO_FEW_POINTS; continue; }  // :134-135
    for (int i = 0; i < 16; ++i) r.T[i] = (double)q.T_cur[i];  // Transform(Eigen::Isometry3f(getFinalTransformation()))  :113-114
    r.fitness = q.fit_n > 0 ? q.fit_sum / (double)q.fit_n : 1.7976931348623157e308;
    r.converged = q.opt.converged; r.outer_iterations = q.opt.nr_iterations; r.inner_iterations = q.opt.line_iterations;
    r.n_correspondences = q.opt.n_pairs_last;
    if (q.active) { r.status = S3D_INTERNAL_ERROR; set_error("NDT round limit reached"); continue; }
    if (!q.opt.converged || r.fitness > cfg.max_fitness_score) { r.status = S3D_NOT_CONVERGED; continue; }  // :107-110
    double ginv[16], delta[16];
    iso_inverse_d(guesses + 16 * p, ginv);
    m4d_mul_d(ginv, r.T, delta);
    const double tn = sqrt(delta[12] * delta[12] + delta[13] * delta[13] + delta[14] * delta[14]);
    r.status = (tn > cfg.max_translation || rotation_angle_of(delta) > cfg.max_rotation) ? S3D_TOO_FAR_FROM_GUESS : S3D_OK;  // :167-172
  }
}

void run_ndt(Workspace& ws, const std::vector<s3d_registration_parameters>& params, const double* guesses, bool direct7, s3d_result* out) {
  std::vector<float> resolution(ws.n_pairs);
  for (uint32_t p = 0; p < ws.n_pairs; ++p) resolution[p] = params[p].resolution;
  run_ndt_grids(ws, kNdtFixedSlots, ws.n_pairs, resolution.data());
  ndt_optimise(ws, params, guesses, direct7, out);
}

void run_ndt_prepared(Workspace& ws, const std::vector<s3d_registration_parameters>& params, const double* guesses, const NdtGrid* grids,
                      bool direct7, s3d_result* out) {
  const uint32_t np = ws.n_pairs;
  ws.ndt_grids.reserve(sizeof(NdtGrid) * std::max<uint32_t>(np, 1));
  ws.h_grids.reserve(sizeof(NdtGrid) * std::max<uint32_t>(np, 1));
  memcpy(ws.h_grids.p, grids, sizeof(NdtGrid) * np);
  S3D_CUDA(cudaMemcpyAsync(ws.ndt_grids.p, ws.h_grids.p, sizeof(NdtGrid) * np, cudaMemcpyHostToDevice, ws.stream));
  ndt_optimise(ws, params, guesses, direct7, out);
}

}  // namespace s3d
