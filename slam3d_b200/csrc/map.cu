// map.cu — the steps around the scan matcher that build patches and maps (SURVEY 8f rank 2/3):
//   PointCloudSensor::transform / getAccumulatedCloud   slam3d/sensor/pcl/PointCloudSensor.cpp:228-256
//   PointCloudSensor::removeOutliers (pcl::RadiusOutlierRemoval, dense-cloud path)             :211-226
//   PointCloudSensor::buildMap = accumulate -> removeOutliers -> downsample                    :301-318
// They re-use the batch plumbing (slots, tiles), the multi-resolution voxel hash (grid.cu) and the VoxelGrid kernels
// (voxel.cu); new here are a streaming rigid transform with concatenation, a fixed-radius neighbour count with early exit
// and an order-preserving compaction.  All are HBM/L2 streaming kernels (16 B in, 16 B out per point).
#include "internal.h"
#include "nn_search.cuh"
#include "sort.cuh"

namespace s3d {

// pcl::transformPointCloud(cloud, out, Matrix4d): double se3 form  x*c0 + (y*c1 + (z*c2 + c3)), cast to float.
// second: optional 16 doubles applied to the (float-rounded) result of the first transform — createCombinedMeasurement's
// transformPointCloud(accumulated, shifted, pose.inverse()) fused into the same pass, with both float roundings kept.
// The one body of both kernels below: the patch path gives the points of s3d_create_combined_measurement bit for bit.
struct Se3d { double t0, t1, t2, t4, t5, t6, t8, t9, t10, t12, t13, t14; };
__device__ __forceinline__ Se3d load_se3d(const double* T) {
  return Se3d{T[0], T[1], T[2], T[4], T[5], T[6], T[8], T[9], T[10], T[12], T[13], T[14]};
}
__device__ __forceinline__ float4 combined_point(float4 p, const Se3d& T, const double* __restrict__ second) {
  const double x = p.x, y = p.y, z = p.z;
  float4 o;
  o.x = (float)__dadd_rn(__dmul_rn(x, T.t0), __dadd_rn(__dmul_rn(y, T.t4), __dadd_rn(__dmul_rn(z, T.t8), T.t12)));
  o.y = (float)__dadd_rn(__dmul_rn(x, T.t1), __dadd_rn(__dmul_rn(y, T.t5), __dadd_rn(__dmul_rn(z, T.t9), T.t13)));
  o.z = (float)__dadd_rn(__dmul_rn(x, T.t2), __dadd_rn(__dmul_rn(y, T.t6), __dadd_rn(__dmul_rn(z, T.t10), T.t14)));
  o.w = 1.0f;
  if (second) {
    const double u = o.x, v = o.y, w = o.z;
    o.x = (float)__dadd_rn(__dmul_rn(u, second[0]), __dadd_rn(__dmul_rn(v, second[4]), __dadd_rn(__dmul_rn(w, second[8]), second[12])));
    o.y = (float)__dadd_rn(__dmul_rn(u, second[1]), __dadd_rn(__dmul_rn(v, second[5]), __dadd_rn(__dmul_rn(w, second[9]), second[13])));
    o.z = (float)__dadd_rn(__dmul_rn(u, second[2]), __dadd_rn(__dmul_rn(v, second[6]), __dadd_rn(__dmul_rn(w, second[10]), second[14])));
  }
  return o;
}

// poses: n_slots x 16 doubles (column-major); out_off: first output index of every slot (clouds are concatenated unpadded).
__global__ void __launch_bounds__(kSortThreads) transform_concat_kernel(const SlotInfo* __restrict__ slots, TileMap tm, const double* __restrict__ poses,
                                                                        const uint32_t* __restrict__ out_off, float4* __restrict__ out,
                                                                        const double* __restrict__ second) {
  const uint32_t t = blockIdx.x;
  const uint32_t slot = tm.tile_slot[t], first = tm.tile_first[t];
  const SlotInfo& si = slots[slot];
  const Se3d T = load_se3d(poses + 16 * (size_t)slot);
#pragma unroll
  for (int j = 0; j < kSortTile / kSortThreads; ++j) {
    const uint32_t e = first + j * kSortThreads + threadIdx.x;
    if (e < si.n_raw) out[out_off[slot] + e] = combined_point(si.raw[e], T, second);
  }
}

// Member m of a multi-patch build: distinct scan `scan` (a slot of the batch), its pose at poses[16 m], its patch's
// patch_pose.inverse() at patch_inv[16 patch] (patch_inv NULL: getAccumulatedCloud), first output index `out`.
struct PatchMember { uint32_t scan, patch, out, reserved; };

// Every patch of a call in one launch: tile t covers points [tile_first, +kSortTile) of member tile_slot[t].  Each scan is read
// from where it was staged once, however many patches it belongs to; the patches land back to back in `out`.
__global__ void __launch_bounds__(kSortThreads) patch_gather_kernel(const SlotInfo* __restrict__ scans, TileMap tm, const PatchMember* __restrict__ members,
                                                                    const double* __restrict__ poses, const double* __restrict__ patch_inv,
                                                                    float4* __restrict__ out) {
  const uint32_t t = blockIdx.x;
  const uint32_t m = tm.tile_slot[t], first = tm.tile_first[t];
  const PatchMember pm = members[m];
  const SlotInfo& si = scans[pm.scan];
  const Se3d T = load_se3d(poses + 16 * (size_t)m);
  const double* second = patch_inv ? patch_inv + 16 * (size_t)pm.patch : nullptr;
#pragma unroll
  for (int j = 0; j < kSortTile / kSortThreads; ++j) {
    const uint32_t e = first + j * kSortThreads + threadIdx.x;
    if (e < si.n_raw) out[pm.out + e] = combined_point(si.raw[e], T, second);
  }
}

// RadiusOutlierRemoval, dense path: keep a point iff at least min_pts + 1 points (itself included) lie within the radius,
// (double)d2 <= radius^2.  One thread per (Morton-sorted) point; the 27-block of the first level whose cells are at least
// `radius` wide covers the whole ball; counting stops as soon as the point is known to stay.
__global__ void __launch_bounds__(256) radius_keep_kernel(const SlotInfo* __restrict__ slots, double r2, float radius, int need, uint8_t* __restrict__ keep) {
  const SlotInfo& si = slots[0];
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= si.n_pts) return;
  const GridView g = make_grid_view(si);
  const float4 q = g.pts[r];
  const uint32_t orig = __float_as_uint(q.w);
  if (g.cap == 0) return;
  int L = 0;
  while (L < g.nlev - 1 && g.h0 * (float)(1 << L) * 0.9999f - g.margin < radius) ++L;
  const float ux = clamp_coord(grid_coord(q.x, g.ox, g.inv_h0)), uy = clamp_coord(grid_coord(q.y, g.oy, g.inv_h0)), uz = clamp_coord(grid_coord(q.z, g.oz, g.inv_h0));
  int cx, cy, cz;
  block_guarantee2(g, ux, uy, uz, L, cx, cy, cz);
  const bool top = L >= g.nlev - 1;
  if (top) cx = cy = cz = 0;
  int count = 0;
  for (int i = 0; i < 27 && count < need; ++i) {
    const int c = cell_order(i);
    uint32_t b, e;
    if (!cell_range(g.table, g.cap, g.nlev, L, cx + c % 3 - 1, cy + (c / 3) % 3 - 1, cz + c / 9 - 1, b, e)) continue;
    for (uint32_t p = b; p < e && count < need; ++p) {
      const float4 v = __ldg(g.pts + p);
      if ((double)dist2_pcl(q.x, q.y, q.z, v.x, v.y, v.z) <= r2) ++count;
    }
  }
  keep[orig] = count >= need ? 1 : 0;
}

// order-preserving compaction of the working cloud by keep[]: per-tile counts, one-warp scan, scatter
__global__ void __launch_bounds__(kSortThreads) keep_count_kernel(const SlotInfo* __restrict__ slots, TileMap tm, const uint8_t* __restrict__ keep,
                                                                   uint32_t* __restrict__ tile_counts) {
  __shared__ uint32_t wsum[8];
  const uint32_t t = blockIdx.x, first = tm.tile_first[t];
  const uint32_t n = slots[0].n_pts;
  uint32_t c = 0;
#pragma unroll
  for (int j = 0; j < kSortTile / kSortThreads; ++j) {
    const uint32_t e = first + threadIdx.x * (kSortTile / kSortThreads) + j;
    if (e < n) c += keep[e];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) { uint32_t s = 0; for (int i = 0; i < 8; ++i) s += wsum[i]; tile_counts[t] = s; }
}

__global__ void keep_scan_kernel(uint32_t n_tiles, uint32_t* __restrict__ tile_counts, uint32_t* __restrict__ total) {
  const int lane = threadIdx.x;
  uint32_t running = 0;
  for (uint32_t b = 0; b < n_tiles; b += 32) {
    const uint32_t t = b + lane;
    const uint32_t v = t < n_tiles ? tile_counts[t] : 0u;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += u; }
    if (t < n_tiles) tile_counts[t] = running + incl - v;
    running += __shfl_sync(0xFFFFFFFFu, incl, 31);
  }
  if (lane == 0) *total = running;
}

__global__ void __launch_bounds__(kSortThreads) keep_scatter_kernel(const SlotInfo* __restrict__ slots, TileMap tm, const uint8_t* __restrict__ keep,
                                                                     const uint32_t* __restrict__ tile_counts, const float4* __restrict__ work,
                                                                     float4* __restrict__ out) {
  __shared__ uint32_t wsum[8];
  const uint32_t t = blockIdx.x, first = tm.tile_first[t];
  const uint32_t n = slots[0].n_pts;
  constexpr int kPer = kSortTile / kSortThreads;
  const uint32_t e0 = first + threadIdx.x * kPer;
  uint32_t c = 0;
#pragma unroll
  for (int j = 0; j < kPer; ++j) if (e0 + j < n) c += keep[e0 + j];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t incl = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += u; }
  if (lane == 31) wsum[w] = incl;
  __syncthreads();
  uint32_t pos = tile_counts[t] + incl - c;
  for (int i = 0; i < w; ++i) pos += wsum[i];
#pragma unroll
  for (int j = 0; j < kPer; ++j) if (e0 + j < n && keep[e0 + j]) out[pos++] = work[e0 + j];
}

// clouds -> one concatenated, transformed cloud in ws.accu (device); returns the number of points
uint32_t run_accumulate(Workspace& ws, const std::vector<const float*>& clouds, const std::vector<uint64_t>& sizes, const double* poses,
                        const double* second) {
  const uint32_t ns = (uint32_t)clouds.size();
  setup_batch(ws, clouds, sizes, 0);
  std::vector<uint32_t> off(ns);
  uint64_t total = 0;
  for (uint32_t s = 0; s < ns; ++s) { off[s] = (uint32_t)total; total += sizes[s]; }
  if (total >= (1ull << 31)) throw CudaError{"map too large: more than 2^31 points"};
  ws.accu.reserve(16 * std::max<uint64_t>(total, 4));
  if (total == 0 || ws.n_tiles == 0) return 0;
  ws.map_aux.reserve(128 * (size_t)(ns + 1) + 4 * (size_t)ns);
  double* d_pose = ws.map_aux.as<double>();
  double* d_second = d_pose + 16 * (size_t)ns;
  uint32_t* d_off = reinterpret_cast<uint32_t*>(d_second + 16);
  S3D_CUDA(cudaMemcpyAsync(d_pose, poses, 128 * (size_t)ns, cudaMemcpyHostToDevice, ws.stream));
  if (second) S3D_CUDA(cudaMemcpyAsync(d_second, second, 128, cudaMemcpyHostToDevice, ws.stream));
  S3D_CUDA(cudaMemcpyAsync(d_off, off.data(), 4 * (size_t)ns, cudaMemcpyHostToDevice, ws.stream));
  TileMap tm{ws.tile_slot.as<uint32_t>(), ws.tile_first.as<uint32_t>(), ws.n_tiles};
  transform_concat_kernel<<<ws.n_tiles, kSortThreads, 0, ws.stream>>>(ws.slots.as<SlotInfo>(), tm, d_pose, d_off, ws.accu.as<float4>(), second ? d_second : nullptr);
  ++ws.launches;
  S3D_CUDA(cudaGetLastError());
  ws.sync();  // `off` and the pageable `poses` must outlive the copies
  return (uint32_t)total;
}

// Patches of s3d_prepare_combined_measurements -> ws.accu (device), patch p at patch_off[p] (n_patches + 1 entries).  Only the
// scans some member references are staged (setup_batch: pinned bounce for pageable memory, device pointers read in place), each
// once; the tables go up in one copy.  Returns after the kernel has finished, so other streams may read ws.accu.
const float4* run_patch_gather(Workspace& ws, const s3d_cloud* scans, const int32_t* member_scan, const double* member_poses,
                               const int32_t* patch_first_member, const double* patch_inv, uint32_t n_patches, std::vector<uint64_t>& patch_off) {
  const uint32_t n_members = (uint32_t)patch_first_member[n_patches];
  std::map<int32_t, uint32_t> slot_of;  // scan index -> slot of the staged batch, in first-use order
  std::vector<const float*> ptrs;
  std::vector<uint64_t> sizes;
  std::vector<PatchMember> members(n_members);
  patch_off.assign(n_patches + 1, 0);
  uint64_t total = 0;
  for (uint32_t p = 0; p < n_patches; ++p) {
    patch_off[p] = total;
    for (int32_t m = patch_first_member[p]; m < patch_first_member[p + 1]; ++m) {
      const int32_t s = member_scan[m];
      auto it = slot_of.find(s);
      if (it == slot_of.end()) {
        it = slot_of.emplace(s, (uint32_t)ptrs.size()).first;
        ptrs.push_back(scans[s].xyzw); sizes.push_back(scans[s].n);
      }
      members[m] = PatchMember{it->second, p, (uint32_t)total, 0};
      total += scans[s].n;
    }
  }
  patch_off[n_patches] = total;
  if (total >= (1ull << 31)) throw CudaError{"patches too large: more than 2^31 points"};
  setup_batch(ws, ptrs, sizes, 0);
  ws.accu.reserve(16 * std::max<uint64_t>(total, 4));
  if (total == 0) return ws.accu.as<float4>();
  std::vector<uint32_t> tile_slot, tile_first;
  for (uint32_t m = 0; m < n_members; ++m)
    for (uint64_t f = 0; f < sizes[members[m].scan]; f += kSortTile) { tile_slot.push_back(m); tile_first.push_back((uint32_t)f); }
  const uint32_t n_tiles = (uint32_t)tile_slot.size();
  // one table block: member poses | patch inverses | members | tile_slot | tile_first
  const size_t b_pose = 128 * (size_t)n_members, b_inv = patch_inv ? 128 * (size_t)n_patches : 0, b_mem = sizeof(PatchMember) * n_members;
  std::vector<char> tab(b_pose + b_inv + b_mem + 8 * (size_t)n_tiles);
  memcpy(tab.data(), member_poses, b_pose);
  if (patch_inv) memcpy(tab.data() + b_pose, patch_inv, b_inv);
  memcpy(tab.data() + b_pose + b_inv, members.data(), b_mem);
  memcpy(tab.data() + b_pose + b_inv + b_mem, tile_slot.data(), 4 * (size_t)n_tiles);
  memcpy(tab.data() + b_pose + b_inv + b_mem + 4 * (size_t)n_tiles, tile_first.data(), 4 * (size_t)n_tiles);
  ws.map_aux.reserve(tab.size());
  char* d = ws.map_aux.as<char>();
  S3D_CUDA(cudaMemcpyAsync(d, tab.data(), tab.size(), cudaMemcpyHostToDevice, ws.stream));
  ws.h2d += tab.size();
  TileMap tm{reinterpret_cast<const uint32_t*>(d + b_pose + b_inv + b_mem), reinterpret_cast<const uint32_t*>(d + b_pose + b_inv + b_mem) + n_tiles, n_tiles};
  patch_gather_kernel<<<n_tiles, kSortThreads, 0, ws.stream>>>(ws.slots.as<SlotInfo>(), tm, reinterpret_cast<const PatchMember*>(d + b_pose + b_inv),
                                                               reinterpret_cast<const double*>(d), patch_inv ? reinterpret_cast<const double*>(d + b_pose) : nullptr,
                                                               ws.accu.as<float4>());
  ++ws.launches;
  S3D_CUDA(cudaGetLastError());
  ws.sync();  // `tab` must outlive the copy, and the prepare pass reads the patches from other streams
  return ws.accu.as<float4>();
}

// RadiusOutlierRemoval of the n points at dev_in (device) into dev_out (device, capacity n); returns the number kept
uint32_t run_radius_filter(Workspace& ws, const float4* dev_in, uint32_t n, double radius, unsigned min_pts, float4* dev_out) {
  setup_batch(ws, {reinterpret_cast<const float*>(dev_in)}, {n}, 0);
  run_voxel(ws, 0.f);  // pass-through: working cloud = input
  run_grid(ws, 0.f);
  ws.map_aux.reserve((size_t)n + 64);
  uint8_t* keep = ws.map_aux.as<uint8_t>();
  S3D_CUDA(cudaMemsetAsync(keep, 0, n, ws.stream));
  const SlotInfo* slots = ws.slots.as<SlotInfo>();
  TileMap tm{ws.tile_slot.as<uint32_t>(), ws.tile_first.as<uint32_t>(), ws.n_tiles};
  radius_keep_kernel<<<(n + 255) / 256, 256, 0, ws.stream>>>(slots, radius * radius, (float)radius, (int)min_pts + 1, keep);
  keep_count_kernel<<<ws.n_tiles, kSortThreads, 0, ws.stream>>>(slots, tm, keep, ws.tile_heads.as<uint32_t>());
  uint32_t* d_total = ws.flags.as<uint32_t>() + 9;
  keep_scan_kernel<<<1, 32, 0, ws.stream>>>(ws.n_tiles, ws.tile_heads.as<uint32_t>(), d_total);
  keep_scatter_kernel<<<ws.n_tiles, kSortThreads, 0, ws.stream>>>(slots, tm, keep, ws.tile_heads.as<uint32_t>(), ws.work.as<float4>(), dev_out);
  ws.launches += 4;
  S3D_CUDA(cudaGetLastError());
  int32_t* hf = ws.h_small.as<int32_t>();
  S3D_CUDA(cudaMemcpyAsync(hf, ws.flags.p, 64, cudaMemcpyDeviceToHost, ws.stream));
  ws.sync();
  ws.d2h += 64;
  check_arena(ws, hf);
  return (uint32_t)hf[9];
}

}  // namespace s3d
