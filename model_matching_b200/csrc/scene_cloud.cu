// scene_cloud.cu -- RGB-D frame -> filtered, down-sampled scene cloud on the device.
//
// Replaces the body of rgbd::load_rgbd_data_sampled (reference src/rgbd.cpp:190-279): depth
// back-projection (:208-225), pcl::VoxelGrid (:227-230), pcl::RadiusOutlierRemoval (:232-236),
// re-projection of each centroid to (row, col), class-probability threshold, depth-normal lookup
// and validity tests (:238-279).  PCL's and OpenCV's own sources are not in the reference tree;
// the operators are restated from their published behaviour (see DESIGN.md, row f1) and the CPU
// oracle restates the same definitions independently, so the two are compared bit for bit.
//
//  * VoxelGrid: leaf key = floor(p / leaf) packed (z,y,x) into 63 bits, stable radix sort of
//    (key, pixel index), one thread per leaf sums its points in pixel order (fp32, sequential, as
//    PCL's accumulation) -> centroids in increasing leaf order.  All zero-depth pixels sit at
//    (0,0,0): they add nothing to a sum, so one representative is sorted and the others only count.
//  * RadiusOutlierRemoval: a centroid's neighbours within r = 2*leaf + 0.005 lie within
//    ceil(r/leaf)+1 leaves per axis; the sorted leaf keys make every (dz,dy) row one binary search
//    plus a linear walk; keep when more than 10 centroids (itself included) are within r.
//  * normals: plane fit over a 9x9 window of the organised cloud (stocs_scene_math.h).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cmath>

#include "stocs_ctx.h"
#include "stocs_scene_math.h"

using namespace stocsm;

namespace {

constexpr long long kOff = 1ll << 20;  // leaf coordinates are offset into [0, 2^21)

__device__ __forceinline__ unsigned long long pack_key(long long ix, long long iy, long long iz) {
  return ((unsigned long long)(iz + kOff) << 42) | ((unsigned long long)(iy + kOff) << 21) | (unsigned long long)(ix + kOff);
}

__global__ void first_zero_kernel(const uint16_t* __restrict__ depth, int n, int* __restrict__ first_zero, int* __restrict__ n_zero) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const bool z = k < n && depth[k] == 0;
  const unsigned b = __ballot_sync(0xffffffffu, z);
  if (z && (threadIdx.x & 31) == (__ffs(b) - 1)) atomicMin(first_zero, k);
  if ((threadIdx.x & 31) == 0 && b) atomicAdd(n_zero, __popc(b));
}

__global__ void voxel_keys_kernel(const float* __restrict__ xyz, const uint16_t* __restrict__ depth, int n, float inv_leaf,
                                  const int* __restrict__ first_zero, unsigned long long* __restrict__ keys,
                                  int* __restrict__ idx, int* __restrict__ n_valid) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const float x = xyz[3 * (size_t)k], y = xyz[3 * (size_t)k + 1], z = xyz[3 * (size_t)k + 2];
  bool valid = isfinite(x) && isfinite(y) && isfinite(z);
  if (valid && depth[k] == 0 && k != *first_zero) valid = false;  // represented by the first zero-depth pixel
  long long ijk[3] = {0, 0, 0};
  if (valid) {
    voxel_coords(x, y, z, inv_leaf, ijk);
    for (int a = 0; a < 3; ++a) if (ijk[a] < -kOff || ijk[a] >= kOff) valid = false;
  }
  keys[k] = valid ? pack_key(ijk[0], ijk[1], ijk[2]) : ~0ull;
  idx[k] = k;
  if (valid) atomicAdd(n_valid, 1);
}

// (list lengths -- valid pixels, voxels -- live in device memory: the host enqueues every stage with
// grids sized by the pixel count and reads the lengths back once, with the result)
__global__ void head_flags_kernel(const unsigned long long* __restrict__ keys, const int* __restrict__ n_valid_p, int* __restrict__ flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *n_valid_p) return;
  flags[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}

__global__ void voxel_starts_kernel(const unsigned long long* __restrict__ keys, const int* __restrict__ flags,
                                    const int* __restrict__ scan, const int* __restrict__ n_valid_p, int* __restrict__ starts,
                                    unsigned long long* __restrict__ ukeys, int* __restrict__ nvox_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n_valid = *n_valid_p;
  if (i == 0) *nvox_out = scan[n_valid];   // flags are zero from n_valid on: the exclusive sum there is the voxel count
  if (i >= n_valid) return;
  if (flags[i]) { starts[scan[i]] = i; ukeys[scan[i]] = keys[i]; }
}

__global__ void centroid_kernel(const float* __restrict__ xyz, const uint16_t* __restrict__ depth, const int* __restrict__ idx,
                                const int* __restrict__ starts, const int* __restrict__ nvox_p, const int* __restrict__ n_valid_p,
                                const int* __restrict__ first_zero, const int* __restrict__ n_zero, float4* __restrict__ cent) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  const int nvox = *nvox_p, n_valid = *n_valid_p;
  if (v >= nvox) return;
  const int s = starts[v], e = (v + 1 < nvox) ? starts[v + 1] : n_valid;
  float sx = 0.f, sy = 0.f, sz = 0.f;
  int count = e - s;
  const int fz = *first_zero;
  for (int t = s; t < e; ++t) {
    const int k = idx[t];
    sx += xyz[3 * (size_t)k]; sy += xyz[3 * (size_t)k + 1]; sz += xyz[3 * (size_t)k + 2];
    if (k == fz && depth[k] == 0) count += *n_zero - 1;
  }
  const float c = (float)count;
  cent[v] = make_float4(sx / c, sy / c, sz / c, 0.f);
}

__global__ void outlier_kernel(const float4* __restrict__ cent, const unsigned long long* __restrict__ ukeys,
                               const int* __restrict__ nvox_p, float r2, int reach, int min_neighbors, int* __restrict__ keep) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  const int nvox = *nvox_p;
  if (v >= nvox) return;
  const float4 p = cent[v];
  const unsigned long long key = ukeys[v];
  const long long ix = (long long)(key & 0x1fffff), iy = (long long)((key >> 21) & 0x1fffff), iz = (long long)(key >> 42);
  int k = 0;
  // keys are sorted (z, y, x): the leaves of one (dz, dy) row are contiguous -> one binary search
  // for the row's first key, then a linear walk
  for (long long dz = -reach; dz <= reach; ++dz)
    for (long long dy = -reach; dy <= reach; ++dy) {
      const long long jy = iy + dy, jz = iz + dz;
      if (jy < 0 || jz < 0 || jy >= 2 * kOff || jz >= 2 * kOff) continue;
      const long long x0 = ix - reach < 0 ? 0 : ix - reach, x1 = ix + reach >= 2 * kOff ? 2 * kOff - 1 : ix + reach;
      const unsigned long long k0 = ((unsigned long long)jz << 42) | ((unsigned long long)jy << 21) | (unsigned long long)x0;
      const unsigned long long k1 = ((unsigned long long)jz << 42) | ((unsigned long long)jy << 21) | (unsigned long long)x1;
      int lo = 0, hi = nvox;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (ukeys[mid] < k0) lo = mid + 1; else hi = mid;
      }
      for (int u = lo; u < nvox && ukeys[u] <= k1; ++u) {
        const float4 q = cent[u];
        const float ex = p.x - q.x, ey = p.y - q.y, ez = p.z - q.z;
        if ((ex * ex + ey * ey) + ez * ez <= r2) ++k;
      }
    }
  keep[v] = (k > min_neighbors) ? 1 : 0;
}

// The per-centroid stage for n_obj probability maps of one frame.  rows holds one int per (object,
// centroid), object-major with n + 1 entries per object (entries from the voxel count on are 0): the
// filter writes 1 where the pair is emitted, one in-place exclusive scan over all n_obj * (n + 1)
// entries turns that into the pair's row of the concatenated output, so that a pair is emitted
// exactly when its entry and the next one differ, and entry k * (n + 1) + n ends object k's rows.
struct FilterArgs {
  const float4* cent; const int* keep; const int* nvox_p; int n; int n_obj; int out_cap;
  const uint16_t* depth; const uint8_t* bgr; const uint16_t* prob; const uint8_t* edge;   // prob: n_obj maps of n
  int W, H; float fx, cx, fy, cy;
  float class_threshold[STOCS_B200_MAX_CLOUD_OBJECTS];
  int* rows;       // n_obj * (n + 1)
  float* nrm;      // nvox * 3 (scratch)
  int* rc;         // nvox * 2
};

__device__ __forceinline__ float class_probability_at(const FilterArgs& a, int k, size_t px) {
  return (float)((double)(float)a.prob[(size_t)k * a.n + px] * (1.0 / 10000));
}

// src/rgbd.cpp:238-279 per centroid: everything but the class test is the same for every object, and the
// normal is computed once, when some object passes
__global__ void filter_kernel(const __grid_constant__ FilterArgs a) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v > a.n) return;
  unsigned pass = 0;   // bit k: object k emits this centroid
  if (v < *a.nvox_p && a.keep[v]) {
    const float4 p = a.cent[v];
    if (!(p.z != p.z) && p.z > 0 && !(p.z > 2.0)) {
      int row, col;
      reproject(p.x, p.y, p.z, a.fx, a.cx, a.fy, a.cy, &row, &col);
      if (row >= 0 && row < a.H && col >= 0 && col < a.W) {  // the reference indexes unchecked here
        const size_t px = (size_t)row * a.W + col;
        for (int k = 0; k < a.n_obj; ++k)
          if (!(class_probability_at(a, k, px) < a.class_threshold[k])) pass |= 1u << k;
        if (pass) {
          float n[3];
          linemod_normal_at(a.depth, a.W, a.H, row, col, a.fx, a.cx, a.fy, a.cy, n);
          const bool bad = (n[0] != n[0]) || (n[1] != n[1]) || (n[2] != n[2]) || (n[0] == 0 && n[1] == 0 && n[2] == 0);
          if (bad) {
            pass = 0;
          } else {
            a.nrm[3 * (size_t)v] = n[0]; a.nrm[3 * (size_t)v + 1] = n[1]; a.nrm[3 * (size_t)v + 2] = n[2];
            a.rc[2 * (size_t)v] = row; a.rc[2 * (size_t)v + 1] = col;
          }
        }
      }
    }
  }
  for (int k = 0; k < a.n_obj; ++k) a.rows[(size_t)k * (a.n + 1) + v] = (pass >> k) & 1;
}

// after the scan: ends[k] = end of object k's rows; every emitted (object, centroid) pair to its row
__global__ void emit_kernel(const __grid_constant__ FilterArgs a, int* __restrict__ ends, float* __restrict__ pos3,
                            float* __restrict__ nrm3, float* __restrict__ rgb3, int* __restrict__ pix2,
                            float* __restrict__ cls, float* __restrict__ edgep) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)a.n + 1;
  if (v < a.n_obj) ends[v] = a.rows[v * stride + a.n];
  if (v >= *a.nvox_p) return;
  int k = 0;
  while (k < a.n_obj && a.rows[k * stride + v] == a.rows[k * stride + v + 1]) ++k;
  if (k == a.n_obj) return;
  const float4 p = a.cent[v];
  const int row = a.rc[2 * (size_t)v], col = a.rc[2 * (size_t)v + 1];
  // Point3D::set_normal normalises (point3d.hpp:43-45)
  const V3 n = normalized(v3(a.nrm[3 * (size_t)v], a.nrm[3 * (size_t)v + 1], a.nrm[3 * (size_t)v + 2]));
  const size_t px = (size_t)row * a.W + col;
  const float r = a.bgr ? (float)a.bgr[3 * px + 2] : 0.f, g = a.bgr ? (float)a.bgr[3 * px + 1] : 0.f,
              b = a.bgr ? (float)a.bgr[3 * px + 0] : 0.f;
  const float e = (float)((255.0 - (double)(a.edge ? a.edge[px] : 0)) / 255.0);
  for (; k < a.n_obj; ++k) {
    const int o = a.rows[k * stride + v];
    if (o == a.rows[k * stride + v + 1]) continue;
    if (o >= a.out_cap) return;   // more points than the caller's buffers hold: reported after the read-back
    pos3[3 * (size_t)o] = p.x; pos3[3 * (size_t)o + 1] = p.y; pos3[3 * (size_t)o + 2] = p.z;
    nrm3[3 * (size_t)o] = n.x; nrm3[3 * (size_t)o + 1] = n.y; nrm3[3 * (size_t)o + 2] = n.z;
    if (rgb3) { rgb3[3 * (size_t)o] = r; rgb3[3 * (size_t)o + 1] = g; rgb3[3 * (size_t)o + 2] = b; }
    pix2[2 * (size_t)o] = row; pix2[2 * (size_t)o + 1] = col;
    cls[o] = class_probability_at(a, k, px);
    if (edgep) edgep[o] = e;
  }
}

// stocs_b200_build_scene_cloud is the one-object case of stocs_b200_build_scene_clouds; `who` prefixes the
// error messages.
int build_scene_clouds(stocs_b200_ctx* ctx, const char* who, const uint16_t* depth, const uint8_t* bgr,
                       const uint16_t* class_probs, const float* class_thresholds, int n_objects, const uint8_t* edge,
                       int W, int H, float fx, float cx, float fy, float cy, float depth_scale, float voxel_size,
                       float* pos3, float* nrm3, float* rgb3, int32_t* pixel_rc, float* class_p, float* edge_p,
                       int64_t cap, int64_t* offsets) {
  // every (object, pixel) entry of the scan and every output row is an int
  const long long rows_needed = (long long)n_objects * ((long long)W * H + 1);
  if (!depth || !class_probs || !class_thresholds || !offsets || n_objects < 1 || n_objects > STOCS_B200_MAX_CLOUD_OBJECTS ||
      W <= 0 || H <= 0 || rows_needed > 0x7fffffffll - 1024 || !(voxel_size > 0) || cap < 0)
    STOCS_FAIL(ctx, STOCS_E_ARG, std::string(who) + ": bad argument");
  for (int k = 0; k <= n_objects; ++k) offsets[k] = 0;
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  const int n = W * H;
  const int nb = (n + 255) / 256;
  DevBuf& d_depth = ctx->pool[POOL_CLOUD_DEPTH];
  DevBuf& d_bgr = ctx->pool[POOL_CLOUD_BGR];
  DevBuf& d_prob = ctx->pool[POOL_CLOUD_PROB];
  DevBuf& d_edge = ctx->pool[POOL_CLOUD_EDGE];
  DevBuf& d_xyz = ctx->pool[POOL_CLOUD_XYZ];
  DevBuf& d_keys_a = ctx->pool[POOL_CLOUD_KEYS_A];
  DevBuf& d_keys_b = ctx->pool[POOL_CLOUD_KEYS_B];
  DevBuf& d_idx_a = ctx->pool[POOL_CLOUD_IDX_A];
  DevBuf& d_idx_b = ctx->pool[POOL_CLOUD_IDX_B];
  DevBuf& d_tmp = ctx->pool[POOL_CLOUD_TMP];
  DevBuf& d_flags = ctx->pool[POOL_CLOUD_FLAGS];
  DevBuf& d_scan = ctx->pool[POOL_CLOUD_SCAN];
  DevBuf& d_starts = ctx->pool[POOL_CLOUD_STARTS];
  DevBuf& d_ukeys = ctx->pool[POOL_CLOUD_UKEYS];
  DevBuf& d_cent = ctx->pool[POOL_CLOUD_CENT];
  DevBuf& d_keep = ctx->pool[POOL_CLOUD_KEEP];
  DevBuf& d_nrm = ctx->pool[POOL_CLOUD_NRM];
  DevBuf& d_rc = ctx->pool[POOL_CLOUD_RC];
  DevBuf& d_out = ctx->pool[POOL_CLOUD_OUT];
#define SC(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) { ctx->err = std::string(#call) + ": " + cudaGetErrorString(_e); return STOCS_E_CUDA; } } while (0)
  SC(d_depth.ensure((size_t)n * 2)); SC(d_prob.ensure((size_t)n_objects * n * 2)); SC(d_xyz.ensure((size_t)n * 12));
  SC(cudaMemcpyAsync(d_depth.p, depth, (size_t)n * 2, cudaMemcpyHostToDevice, st));
  SC(cudaMemcpyAsync(d_prob.p, class_probs, (size_t)n_objects * n * 2, cudaMemcpyHostToDevice, st));
  if (bgr) { SC(d_bgr.ensure((size_t)n * 3)); SC(cudaMemcpyAsync(d_bgr.p, bgr, (size_t)n * 3, cudaMemcpyHostToDevice, st)); }
  if (edge) { SC(d_edge.ensure((size_t)n)); SC(cudaMemcpyAsync(d_edge.p, edge, (size_t)n, cudaMemcpyHostToDevice, st)); }
  int rc = stocs_launch_backproject(ctx, d_depth.as<uint16_t>(), nullptr, W, H, fx, cx, fy, cy, depth_scale, d_xyz.as<float>(), nullptr, st);
  if (rc) return rc;
  // device counters: first_zero, n_zero, n_valid, n_vox, then the end of each object's rows (emit_kernel)
  int* d_cnt = ctx->scratch()->cloud;
  int init[3] = {0x7fffffff, 0, 0};
  SC(cudaMemcpyAsync(d_cnt, init, 12, cudaMemcpyHostToDevice, st));
  first_zero_kernel<<<nb, 256, 0, st>>>(d_depth.as<uint16_t>(), n, d_cnt, d_cnt + 1);
  SC(d_keys_a.ensure((size_t)n * 8)); SC(d_keys_b.ensure((size_t)n * 8)); SC(d_idx_a.ensure((size_t)n * 4)); SC(d_idx_b.ensure((size_t)n * 4));
  voxel_keys_kernel<<<nb, 256, 0, st>>>(d_xyz.as<float>(), d_depth.as<uint16_t>(), n, 1.0f / voxel_size, d_cnt,
                                        d_keys_a.as<unsigned long long>(), d_idx_a.as<int>(), d_cnt + 2);
  size_t tb = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tb, d_keys_a.as<unsigned long long>(), d_keys_b.as<unsigned long long>(), d_idx_a.as<int>(),
                                  d_idx_b.as<int>(), n, 0, 64, st);
  SC(d_tmp.ensure(tb));
  cub::DeviceRadixSort::SortPairs(d_tmp.p, tb, d_keys_a.as<unsigned long long>(), d_keys_b.as<unsigned long long>(), d_idx_a.as<int>(),
                                  d_idx_b.as<int>(), n, 0, 64, st);
  // ---- every later stage is enqueued against the pixel count n; the list lengths stay on the device
  int* d_nvalid = d_cnt + 2;
  int* d_nvox = d_cnt + 3;
  const unsigned long long* keys = d_keys_b.as<unsigned long long>();
  const int* idx = d_idx_b.as<int>();
  const int n_rows = n_objects * (n + 1);   // the filter's flags, one per (object, pixel)
  SC(d_flags.ensure((size_t)n_rows * 4)); SC(d_scan.ensure((size_t)(n + 1) * 4));
  SC(d_starts.ensure((size_t)n * 4)); SC(d_ukeys.ensure((size_t)n * 8)); SC(d_cent.ensure((size_t)n * 16));
  SC(d_keep.ensure((size_t)(n + 1) * 4)); SC(d_nrm.ensure((size_t)n * 12)); SC(d_rc.ensure((size_t)n * 8));
  SC(cudaMemsetAsync(d_flags.p, 0, (size_t)(n + 1) * 4, st));
  head_flags_kernel<<<nb, 256, 0, st>>>(keys, d_nvalid, d_flags.as<int>());
  size_t tb2 = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tb2, d_flags.as<int>(), d_scan.as<int>(), n + 1, st);
  SC(d_tmp.ensure(tb2));
  cub::DeviceScan::ExclusiveSum(d_tmp.p, tb2, d_flags.as<int>(), d_scan.as<int>(), n + 1, st);
  voxel_starts_kernel<<<nb, 256, 0, st>>>(keys, d_flags.as<int>(), d_scan.as<int>(), d_nvalid, d_starts.as<int>(),
                                          d_ukeys.as<unsigned long long>(), d_nvox);
  const int nxb = (n + 127) / 128;
  centroid_kernel<<<nxb, 128, 0, st>>>(d_xyz.as<float>(), d_depth.as<uint16_t>(), idx, d_starts.as<int>(), d_nvox, d_nvalid, d_cnt,
                                       d_cnt + 1, d_cent.as<float4>());
  // src/rgbd.cpp:234: setRadiusSearch(double(2*voxel_size) + 0.005); the search compares squared
  // distances with float(radius * radius) (pcl::KdTreeFLANN::radiusSearch)
  const double radius = (double)(2 * voxel_size) + 0.005;
  const float r2 = (float)(radius * radius);
  const int reach = (int)std::ceil(radius / (double)voxel_size) + 1;
  outlier_kernel<<<nxb, 128, 0, st>>>(d_cent.as<float4>(), d_ukeys.as<unsigned long long>(), d_nvox, r2, reach, 10, d_keep.as<int>());
  // one flag per (object, centroid), scanned in place into output rows (see FilterArgs)
  const long long out_cap = cap < (long long)n_objects * n ? cap : (long long)n_objects * n;
  FilterArgs fa;
  fa.cent = d_cent.as<float4>(); fa.keep = d_keep.as<int>(); fa.nvox_p = d_nvox; fa.n = n; fa.n_obj = n_objects;
  fa.out_cap = (int)out_cap;
  fa.depth = d_depth.as<uint16_t>();
  fa.bgr = bgr ? d_bgr.as<uint8_t>() : nullptr; fa.prob = d_prob.as<uint16_t>(); fa.edge = edge ? d_edge.as<uint8_t>() : nullptr;
  fa.W = W; fa.H = H; fa.fx = fx; fa.cx = cx; fa.fy = fy; fa.cy = cy;
  for (int k = 0; k < STOCS_B200_MAX_CLOUD_OBJECTS; ++k) fa.class_threshold[k] = k < n_objects ? class_thresholds[k] : 0.f;
  fa.rows = d_flags.as<int>(); fa.nrm = d_nrm.as<float>(); fa.rc = d_rc.as<int>();
  filter_kernel<<<(n + 1 + 127) / 128, 128, 0, st>>>(fa);
  size_t tb3 = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tb3, fa.rows, n_rows, st);
  SC(d_tmp.ensure(tb3));
  cub::DeviceScan::ExclusiveSum(d_tmp.p, tb3, fa.rows, n_rows, st);
  // out: pos3 | nrm3 | rgb3 | pix2 | cls | edge, each with room for out_cap points
  const size_t oc = (size_t)(out_cap > 0 ? out_cap : 1);
  SC(d_out.ensure(oc * (12 + 12 + 12 + 8 + 4 + 4)));
  float* o_pos = d_out.as<float>();
  float* o_nrm = o_pos + 3 * oc;
  float* o_rgb = o_nrm + 3 * oc;
  int* o_pix = (int*)(o_rgb + 3 * oc);
  float* o_cls = (float*)(o_pix + 2 * oc);
  float* o_edge = o_cls + oc;
  int* d_ends = d_cnt + 4;
  emit_kernel<<<nxb, 128, 0, st>>>(fa, d_ends, o_pos, o_nrm, o_rgb, o_pix, o_cls, o_edge);
  SC(cudaGetLastError());
  // read-back: the voxel count and every object's end, and -- in the same queue, before anything is
  // known -- as many points as the previous call's estimate below; a frame that emits more fetches the
  // rest afterwards
  uint32_t* h_len = ctx->h_index_counts + 8;   // page-locked: {voxels, end of object 0, .., end of object K-1}
  SC(cudaMemcpyAsync(h_len, d_nvox, (size_t)(1 + n_objects) * 4, cudaMemcpyDeviceToHost, st));
  const bool have_out = pos3 && nrm3 && pixel_rc && class_p;
  // the previous voxel count bounds what one object of a frame like the previous one emits; with several
  // objects, the previous call's points plus that much again
  const long long prev_vox = ctx->counters[CTR_CLOUD_VOXELS];
  long long guess = have_out ? std::min((long long)n_objects * prev_vox, ctx->cloud_last_points + prev_vox) : 0;
  if (guess > out_cap) guess = out_cap;
  auto fetch = [&](long long from, long long to) -> cudaError_t {
    const size_t c = (size_t)(to - from);
    cudaError_t e = cudaMemcpyAsync(pos3 + 3 * from, o_pos + 3 * from, c * 12, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(nrm3 + 3 * from, o_nrm + 3 * from, c * 12, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && rgb3) e = cudaMemcpyAsync(rgb3 + 3 * from, o_rgb + 3 * from, c * 12, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(pixel_rc + 2 * from, o_pix + 2 * from, c * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(class_p + from, o_cls + from, c * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && edge_p) e = cudaMemcpyAsync(edge_p + from, o_edge + from, c * 4, cudaMemcpyDeviceToHost, st);
    return e;
  };
  if (guess > 0) SC(fetch(0, guess));
  SC(cudaStreamSynchronize(st));
  const long long nvox = (long long)h_len[0];
  for (int k = 0; k < n_objects; ++k) offsets[k + 1] = (int64_t)h_len[1 + k];
  const long long n_emit = offsets[n_objects];
  ctx->counters[CTR_CLOUD_VOXELS] = nvox;
  ctx->cloud_last_points = n_emit;
  if (n_emit > cap) STOCS_FAIL(ctx, STOCS_E_CAPACITY, std::string(who) + ": output capacity too small");
  if (n_emit > 0 && !have_out) STOCS_FAIL(ctx, STOCS_E_ARG, std::string(who) + ": output pointer is NULL");
  if (n_emit > guess) {
    SC(fetch(guess, n_emit));
    SC(cudaStreamSynchronize(st));
  }
#undef SC
  return STOCS_OK;
}

}  // namespace

extern "C" int stocs_b200_build_scene_clouds(stocs_b200_ctx* ctx, const uint16_t* depth, const uint8_t* bgr,
                                             const uint16_t* class_probs, const float* class_thresholds, int n_objects,
                                             const uint8_t* edge, int W, int H, float fx, float cx, float fy, float cy,
                                             float depth_scale, float voxel_size, float* pos3, float* nrm3, float* rgb3,
                                             int32_t* pixel_rc, float* class_p, float* edge_p, int64_t cap, int64_t* offsets) {
  if (!ctx) return STOCS_E_ARG;
  return build_scene_clouds(ctx, "build_scene_clouds", depth, bgr, class_probs, class_thresholds, n_objects, edge, W, H, fx,
                            cx, fy, cy, depth_scale, voxel_size, pos3, nrm3, rgb3, pixel_rc, class_p, edge_p, cap, offsets);
}

extern "C" int stocs_b200_build_scene_cloud(stocs_b200_ctx* ctx, const uint16_t* depth, const uint8_t* bgr,
                                            const uint16_t* class_prob, const uint8_t* edge, int W, int H, float fx,
                                            float cx, float fy, float cy, float depth_scale, float voxel_size,
                                            float class_threshold, float* pos3, float* nrm3, float* rgb3,
                                            int32_t* pixel_rc, float* class_p, float* edge_p, int64_t cap, int64_t* n_out) {
  if (!ctx) return STOCS_E_ARG;
  if (!n_out) STOCS_FAIL(ctx, STOCS_E_ARG, "build_scene_cloud: bad argument");
  int64_t offsets[2] = {0, 0};
  const int rc = build_scene_clouds(ctx, "build_scene_cloud", depth, bgr, class_prob, &class_threshold, 1, edge, W, H, fx,
                                    cx, fy, cy, depth_scale, voxel_size, pos3, nrm3, rgb3, pixel_rc, class_p, edge_p, cap,
                                    offsets);
  *n_out = offsets[1];
  return rc;
}
