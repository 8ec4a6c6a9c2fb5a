// ppf_table.cu -- compact point-pair-feature table of the model, built on the device.
//
// Replaces the pair loop of stocs::pre_process_model (reference src/stocs.cpp:62-78),
// rgbd::ppf_map_insert (src/rgbd.cpp:123-154) and PPFMapType (include/rgbd.hpp:23): see
// ppf_device.cuh for the representation.  O(M^2) ppf_compute calls, one 64-bit radix sort.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <cmath>

#include "ppf_device.cuh"
#include "stocs_ctx.h"

using namespace stocsm;

namespace {

__global__ void ppf_pairs_kernel(const float* __restrict__ pos3, const float4* __restrict__ nrm4, int M, int n1,
                                 int na, int tr, int rot, unsigned long long* __restrict__ keys,
                                 uint32_t* __restrict__ counts) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)M * M) return;
  const int id1 = (int)(t / M), id2 = (int)(t - (long long)id1 * M);
  if (id1 == id2) { keys[t] = ~0ull; return; }
  const V3 p1 = v3(pos3[3 * id1], pos3[3 * id1 + 1], pos3[3 * id1 + 2]);
  const V3 p2 = v3(pos3[3 * id2], pos3[3 * id2 + 1], pos3[3 * id2 + 2]);
  const float4 a = nrm4[id1], b = nrm4[id2];
  const Ppf4 f = ppf_compute(p1, v3(a.x, a.y, a.z), p2, v3(b.x, b.y, b.z), tr, rot);
  int b1 = f.f[0] / tr, b2 = f.f[1] / rot, b3 = f.f[2] / rot, b4 = f.f[3] / rot;
  if (b1 < 0 || b1 >= n1 || b2 < 0 || b2 >= na || b3 < 0 || b3 >= na || b4 < 0 || b4 >= na) {
    keys[t] = ~0ull;  // NaN normals etc.: the reference's int(NaN) is undefined; such pairs are dropped
    return;
  }
  const uint32_t bin = (uint32_t)(((b1 * na + b2) * na + b3) * na + b4);
  keys[t] = ((unsigned long long)bin << 32) | ((unsigned long long)id1 << 16) | (unsigned long long)id2;
  atomicAdd(&counts[bin], 1u);
}

// the same sort keys from a caller-provided table (key4 = own-bin key in mm / degrees, pair = ids);
// *bad counts entries that do not fit this model / discretisation
__global__ void ppf_from_list_kernel(const int* __restrict__ keys4, const int* __restrict__ pairs2, long long n, int M,
                                     int n1, int na, int tr, int rot, unsigned long long* __restrict__ keys,
                                     uint32_t* __restrict__ counts, unsigned long long* __restrict__ bad) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int k1 = keys4[4 * t], k2 = keys4[4 * t + 1], k3 = keys4[4 * t + 2], k4 = keys4[4 * t + 3];
  const int id1 = pairs2[2 * t], id2 = pairs2[2 * t + 1];
  const int b1 = k1 / tr, b2 = k2 / rot, b3 = k3 / rot, b4 = k4 / rot;
  const bool ok = k1 >= 0 && k2 >= 0 && k3 >= 0 && k4 >= 0 && k1 % tr == 0 && k2 % rot == 0 && k3 % rot == 0 && k4 % rot == 0 &&
                  b1 < n1 && b2 < na && b3 < na && b4 < na && id1 >= 0 && id1 < M && id2 >= 0 && id2 < M && id1 != id2;
  if (!ok) { keys[t] = ~0ull; atomicAdd(bad, 1ull); return; }
  const uint32_t bin = (uint32_t)(((b1 * na + b2) * na + b3) * na + b4);
  keys[t] = ((unsigned long long)bin << 32) | ((unsigned long long)id1 << 16) | (unsigned long long)id2;
  atomicAdd(&counts[bin], 1u);
}

__global__ void ppf_strip_kernel(const unsigned long long* __restrict__ keys, long long n, uint32_t* __restrict__ pairs) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) pairs[t] = (uint32_t)(keys[t] & 0xffffffffull);
}

// one thread per own bin: a non-empty bin sets the bits of the (<= 128) keys it was inserted under
__global__ void ppf_keybits_kernel(const uint32_t* __restrict__ bin_start, int n1, int na, int tr,
                                   uint32_t* __restrict__ keybits, unsigned long long* __restrict__ nkeys) {
  const long long nb = (long long)n1 * na * na * na;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nb) return;
  if (bin_start[t + 1] == bin_start[t]) return;
  atomicAdd(nkeys, 1ull);
  int r = (int)t;
  const int b4 = r % na; r /= na;
  const int b3 = r % na; r /= na;
  const int b2 = r % na; r /= na;
  const int b1 = r;
  const int nk = na + 1;
  for (int a = -1; a <= 0; ++a) {
    const int k1 = b1 + a;
    if (k1 * tr <= 5) continue;  // "distances less than 5mm are not allowed" (rgbd.cpp:136)
    for (int b = -2; b <= 1; ++b) {
      const int k2 = b2 + b;
      if (k2 < 0) continue;
      for (int c = -2; c <= 1; ++c) {
        const int k3 = b3 + c;
        if (k3 < 0) continue;
        for (int d = -2; d <= 1; ++d) {
          const int k4 = b4 + d;
          if (k4 < 0) continue;
          const uint32_t bit = (uint32_t)(((k1 * nk + k2) * nk + k3) * nk + k4);
          atomicOr(&keybits[bit >> 5], 1u << (bit & 31));
        }
      }
    }
  }
}

__global__ void ppf_count_bits_kernel(const uint32_t* __restrict__ bits, long long nwords, unsigned long long* __restrict__ out) {
  unsigned long long c = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nwords; i += (long long)gridDim.x * blockDim.x)
    c += __popc(bits[i]);
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

__global__ void ppf_export_kernel(const uint32_t* __restrict__ bin_start, const uint32_t* __restrict__ pairs, int n1, int na,
                                  int tr, int rot, int* __restrict__ keys4, int* __restrict__ pairs2) {
  const long long nb = (long long)n1 * na * na * na;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nb) return;
  const uint32_t s = bin_start[t], e = bin_start[t + 1];
  if (s == e) return;
  int r = (int)t;
  const int b4 = r % na; r /= na;
  const int b3 = r % na; r /= na;
  const int b2 = r % na; r /= na;
  for (uint32_t k = s; k < e; ++k) {
    keys4[4 * (size_t)k] = r * tr; keys4[4 * (size_t)k + 1] = b2 * rot; keys4[4 * (size_t)k + 2] = b3 * rot; keys4[4 * (size_t)k + 3] = b4 * rot;
    pairs2[2 * (size_t)k] = (int)(pairs[k] >> 16); pairs2[2 * (size_t)k + 1] = (int)(pairs[k] & 0xffffu);
  }
}

// map lookup for the C ABI: gather the source bins of one key into out[], count in *n
__global__ void ppf_gather_kernel(PpfView v, Ppf4 key, uint32_t* __restrict__ out, long long cap,
                                  long long* __restrict__ n_out) {
  __shared__ uint32_t s_start[128], s_cnt[128], s_off[129];
  const int j = threadIdx.x;  // 128 threads
  const bool valid = !(key.f[0] <= 5 || key.f[1] < 0 || key.f[2] < 0 || key.f[3] < 0) &&
                     key.f[0] % v.tr == 0 && key.f[1] % v.rot == 0 && key.f[2] % v.rot == 0 && key.f[3] % v.rot == 0;
  uint32_t bin = 0xffffffffu;
  if (valid) bin = ppf_source_bin(v, key.f[0] / v.tr, key.f[1] / v.rot, key.f[2] / v.rot, key.f[3] / v.rot, j);
  s_start[j] = 0; s_cnt[j] = 0;
  if (bin != 0xffffffffu) { s_start[j] = v.bin_start[bin]; s_cnt[j] = v.bin_start[bin + 1] - s_start[j]; }
  __syncthreads();
  if (j == 0) {
    uint32_t acc = 0;
    for (int k = 0; k < 128; ++k) { s_off[k] = acc; acc += s_cnt[k]; }
    s_off[128] = acc;
    *n_out = acc ? (long long)acc : -1ll;
  }
  __syncthreads();
  for (int k = 0; k < 128; ++k)
    for (uint32_t e = j; e < s_cnt[k]; e += 128)
      if ((long long)(s_off[k] + e) < cap) out[s_off[k] + e] = v.pairs[s_start[k] + e];
}

}  // namespace

PpfView stocs_ppf_view(const stocs_b200_ctx* ctx) {
  PpfView v;
  v.bin_start = ctx->d_ppf_bin_start.as<uint32_t>();
  v.pairs = ctx->d_ppf_pairs.as<uint32_t>();
  v.keybits = ctx->d_ppf_keybits.as<uint32_t>();
  v.n1 = ctx->ppf.n1; v.na = ctx->ppf.na; v.tr = ctx->ppf.tr; v.rot = ctx->ppf.rot;
  return v;
}

// expects ctx->d_tmp = raw (un-centred) model pos3, ctx->d_mnrm4 = normals -- or, with list_n >= 0, a
// caller-provided table (device arrays d_keys4 / d_pairs2 of list_n entries) instead of the pair loop
static int build_ppf_table(stocs_b200_ctx* ctx, const int* d_keys4, const int* d_pairs2, long long list_n) {
  const int M = ctx->M;
  cudaStream_t st = ctx->stream;
  // bound on f1: the model diagonal (centred AABB == raw AABB extents up to rounding; add slack)
  float mn[3] = {1e30f, 1e30f, 1e30f}, mx[3] = {-1e30f, -1e30f, -1e30f};
  for (int i = 0; i < M; ++i)
    for (int k = 0; k < 3; ++k) {
      float c = ctx->h_mpos[3 * (size_t)i + k];
      if (c < mn[k]) mn[k] = c;
      if (c > mx[k]) mx[k] = c;
    }
  double diag = std::sqrt((double)(mx[0] - mn[0]) * (mx[0] - mn[0]) + (double)(mx[1] - mn[1]) * (mx[1] - mn[1]) +
                          (double)(mx[2] - mn[2]) * (mx[2] - mn[2]));
  if (!(diag < 100.0)) STOCS_FAIL(ctx, STOCS_E_ARG, "upload_model: model extent must be finite and < 100 m");
  const int tr = ctx->tr, rot = ctx->rot;
  const int n1 = (int)(diag * 1000.0 * 1.001) / tr + 3;
  const int na = 180 / rot + 2;
  const long long nbins = (long long)n1 * na * na * na;
  const long long nkeybits = (long long)(n1 + 1) * (na + 1) * (na + 1) * (na + 1);
  if (nbins > (1ll << 30)) STOCS_FAIL(ctx, STOCS_E_ARG, "upload_model: PPF bin space too large (coarser discretisation needed)");
  ctx->ppf.n1 = n1; ctx->ppf.na = na; ctx->ppf.tr = tr; ctx->ppf.rot = rot;
  const long long MM = list_n >= 0 ? (list_n > 0 ? list_n : 1) : (long long)M * M;
  STOCS_CUDA(ctx, ctx->d_ppf_bin_start.ensure((size_t)(nbins + 1) * 4));
  STOCS_CUDA(ctx, ctx->d_ppf_keybits.ensure((size_t)((nkeybits + 31) / 32) * 4));
  STOCS_CUDA(ctx, ctx->d_work.ensure((size_t)(nbins + 1) * 4));
  DevBuf &keys_a = ctx->pool[POOL_PPF_KEYS_A], &keys_b = ctx->pool[POOL_PPF_KEYS_B], &cub_tmp = ctx->pool[POOL_PPF_CUB_TMP];
  STOCS_CUDA(ctx, keys_a.ensure((size_t)MM * 8));
  STOCS_CUDA(ctx, keys_b.ensure((size_t)MM * 8));
  uint32_t* counts = ctx->d_work.as<uint32_t>();
  STOCS_CUDA(ctx, cudaMemsetAsync(counts, 0, (size_t)(nbins + 1) * 4, st));
  STOCS_CUDA(ctx, cudaMemsetAsync(ctx->d_ppf_keybits.p, 0, (size_t)((nkeybits + 31) / 32) * 4, st));
  if (list_n >= 0) {
    unsigned long long* d_bad = &ctx->scratch()->ppf_bad;
    STOCS_CUDA(ctx, cudaMemsetAsync(d_bad, 0, 8, st));
    STOCS_CUDA(ctx, cudaMemsetAsync(keys_a.p, 0xff, (size_t)MM * 8, st));
    if (list_n > 0)
      ppf_from_list_kernel<<<(unsigned)((list_n + 255) / 256), 256, 0, st>>>(d_keys4, d_pairs2, list_n, M, n1, na, tr, rot,
                                                                             keys_a.as<unsigned long long>(), counts, d_bad);
    unsigned long long bad = 0;
    STOCS_CUDA(ctx, cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, st));
    STOCS_CUDA(ctx, cudaStreamSynchronize(st));
    if (bad) STOCS_FAIL(ctx, STOCS_E_ARG, "upload_ppf_table: " + std::to_string(bad) + " entries do not fit this model / discretisation "
                                          "(ids >= |M|, keys off the bin lattice or beyond the model diagonal)");
  } else {
    ppf_pairs_kernel<<<(unsigned)((MM + 255) / 256), 256, 0, st>>>(ctx->d_tmp.as<float>(), ctx->d_mnrm4.as<float4>(), M, n1,
                                                                    na, tr, rot, keys_a.as<unsigned long long>(), counts);
  }
  size_t tb = 0, tb2 = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, tb, keys_a.as<unsigned long long>(), keys_b.as<unsigned long long>(), (int)MM, 0, 64, st);
  cub::DeviceScan::ExclusiveSum(nullptr, tb2, counts, ctx->d_ppf_bin_start.as<uint32_t>(), (int)(nbins + 1), st);
  STOCS_CUDA(ctx, cub_tmp.ensure(tb > tb2 ? tb : tb2));
  cub::DeviceRadixSort::SortKeys(cub_tmp.p, tb, keys_a.as<unsigned long long>(), keys_b.as<unsigned long long>(), (int)MM, 0, 64, st);
  cub::DeviceScan::ExclusiveSum(cub_tmp.p, tb2, counts, ctx->d_ppf_bin_start.as<uint32_t>(), (int)(nbins + 1), st);
  uint32_t npairs = 0;
  STOCS_CUDA(ctx, cudaMemcpyAsync(&npairs, ctx->d_ppf_bin_start.as<uint32_t>() + nbins, 4, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  STOCS_CUDA(ctx, ctx->d_ppf_pairs.ensure((size_t)(npairs ? npairs : 1) * 4));
  if (npairs)
    ppf_strip_kernel<<<(npairs + 255) / 256, 256, 0, st>>>(keys_b.as<unsigned long long>(), npairs, ctx->d_ppf_pairs.as<uint32_t>());
  unsigned long long* d_nkeys = &ctx->scratch()->ppf_nkeys;
  STOCS_CUDA(ctx, cudaMemsetAsync(d_nkeys, 0, 8, st));
  ppf_keybits_kernel<<<(unsigned)((nbins + 255) / 256), 256, 0, st>>>(ctx->d_ppf_bin_start.as<uint32_t>(), n1, na, tr,
                                                                       ctx->d_ppf_keybits.as<uint32_t>(), d_nkeys);
  unsigned long long nk = 0;
  STOCS_CUDA(ctx, cudaMemcpyAsync(&nk, d_nkeys, 8, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  STOCS_CUDA(ctx, cudaGetLastError());
  ctx->ppf.npairs = npairs;
  ctx->ppf.nkeys = (int64_t)nk;
  STOCS_CUDA(ctx, cudaMemsetAsync(d_nkeys, 0, 8, st));
  ppf_count_bits_kernel<<<64, 256, 0, st>>>(ctx->d_ppf_keybits.as<uint32_t>(), (nkeybits + 31) / 32, d_nkeys);
  STOCS_CUDA(ctx, cudaMemcpyAsync(&nk, d_nkeys, 8, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->ppf.nexpanded = (int64_t)nk;
  return STOCS_OK;
}

int stocs_build_ppf_table(stocs_b200_ctx* ctx) { return build_ppf_table(ctx, nullptr, nullptr, -1); }

extern "C" {

// The table a caller preloaded (reference: ppf_map_preloaded, src/stocs.cpp:94) replaces the one
// upload_model derived from the points.  A table that cannot belong to this model is an error, never
// silently ignored.  On failure the context keeps no PPF table (M is reset: upload the model again).
int stocs_b200_upload_ppf_table(stocs_b200_ctx* ctx, const int32_t* keys4, const int32_t* pairs2, int64_t n,
                                int tr_discretization, int rot_discretization, int num_model_points) {
  if (!ctx) return STOCS_E_ARG;
  if (ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "upload_ppf_table: upload_model first");
  if (n < 0 || (n > 0 && (!keys4 || !pairs2))) STOCS_FAIL(ctx, STOCS_E_ARG, "upload_ppf_table: bad argument");
  if (tr_discretization != ctx->tr || rot_discretization != ctx->rot)
    STOCS_FAIL(ctx, STOCS_E_ARG, "upload_ppf_table: the table was built with discretisation (" + std::to_string(tr_discretization) + ", " +
                                     std::to_string(rot_discretization) + "), the estimator uses (" + std::to_string(ctx->tr) + ", " +
                                     std::to_string(ctx->rot) + ")");
  if (num_model_points != ctx->M)
    STOCS_FAIL(ctx, STOCS_E_ARG, "upload_ppf_table: the table was built for " + std::to_string(num_model_points) +
                                     " model points, the uploaded model has " + std::to_string(ctx->M));
  if (n >= (1ll << 31)) STOCS_FAIL(ctx, STOCS_E_ARG, "upload_ppf_table: too many entries");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  DevBuf dk, dp;
  cudaError_t e = dk.ensure((size_t)(n ? n : 1) * 16);
  if (e == cudaSuccess) e = dp.ensure((size_t)(n ? n : 1) * 8);
  if (e == cudaSuccess && n) e = cudaMemcpyAsync(dk.p, keys4, (size_t)n * 16, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess && n) e = cudaMemcpyAsync(dp.p, pairs2, (size_t)n * 8, cudaMemcpyHostToDevice, st);
  int rc = STOCS_OK;
  if (e != cudaSuccess) { ctx->err = std::string("upload_ppf_table: ") + cudaGetErrorString(e); rc = STOCS_E_CUDA; }
  if (rc == STOCS_OK) rc = build_ppf_table(ctx, dk.as<int>(), dp.as<int>(), n);
  cudaStreamSynchronize(st);
  dk.release(); dp.release();
  if (rc != STOCS_OK) { ctx->M = 0; ctx->ppf = PpfTableDesc{}; }
  return rc;
}

int stocs_b200_ppf_num_pairs(stocs_b200_ctx* ctx, int64_t* own_bin_pairs, int64_t* own_bin_keys) {
  if (!ctx) return STOCS_E_ARG;
  if (ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "ppf: upload_model first");
  if (own_bin_pairs) *own_bin_pairs = ctx->ppf.npairs;
  if (own_bin_keys) *own_bin_keys = ctx->ppf.nkeys;
  return STOCS_OK;
}

int stocs_b200_ppf_num_expanded_keys(stocs_b200_ctx* ctx, int64_t* expanded_keys) {
  if (!ctx || !expanded_keys) return STOCS_E_ARG;
  if (ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "ppf: upload_model first");
  *expanded_keys = ctx->ppf.nexpanded;
  return STOCS_OK;
}

int stocs_b200_ppf_export(stocs_b200_ctx* ctx, int32_t* keys4, int32_t* pairs2, int64_t cap, int64_t* n) {
  if (!ctx || !n) return STOCS_E_ARG;
  if (ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "ppf: upload_model first");
  *n = ctx->ppf.npairs;
  if (!keys4 || !pairs2) return STOCS_OK;
  if (cap < ctx->ppf.npairs) STOCS_FAIL(ctx, STOCS_E_CAPACITY, "ppf_export: capacity too small");
  if (ctx->ppf.npairs == 0) return STOCS_OK;
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  DevBuf dk, dp;
  STOCS_CUDA(ctx, dk.ensure((size_t)ctx->ppf.npairs * 16));
  STOCS_CUDA(ctx, dp.ensure((size_t)ctx->ppf.npairs * 8));
  const long long nb = (long long)ctx->ppf.n1 * ctx->ppf.na * ctx->ppf.na * ctx->ppf.na;
  ppf_export_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, st>>>(ctx->d_ppf_bin_start.as<uint32_t>(), ctx->d_ppf_pairs.as<uint32_t>(),
                                                                  ctx->ppf.n1, ctx->ppf.na, ctx->ppf.tr, ctx->ppf.rot, dk.as<int>(), dp.as<int>());
  STOCS_CUDA(ctx, cudaMemcpyAsync(keys4, dk.p, (size_t)ctx->ppf.npairs * 16, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(pairs2, dp.p, (size_t)ctx->ppf.npairs * 8, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  dk.release(); dp.release();
  return STOCS_OK;
}

int stocs_b200_ppf_lookup(stocs_b200_ctx* ctx, const int32_t* key4, int32_t* pairs2, int64_t cap, int64_t* count) {
  if (!ctx) return STOCS_E_ARG;
  if (ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "ppf: upload_model first");
  if (!key4 || !count || cap < 0) STOCS_FAIL(ctx, STOCS_E_ARG, "ppf_lookup: bad argument");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  Ppf4 key;
  for (int k = 0; k < 4; ++k) key.f[k] = key4[k];
  const long long maxn = ctx->ppf.npairs > 0 ? ctx->ppf.npairs : 1;
  DevBuf a, b, tmp;
  STOCS_CUDA(ctx, a.ensure((size_t)maxn * 4));
  STOCS_CUDA(ctx, b.ensure((size_t)maxn * 4));
  long long* d_n = &ctx->scratch()->ppf_lookup_n;
  ppf_gather_kernel<<<1, 128, 0, st>>>(stocs_ppf_view(ctx), key, a.as<uint32_t>(), maxn, d_n);
  long long n = 0;
  STOCS_CUDA(ctx, cudaMemcpyAsync(&n, d_n, 8, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  *count = n;
  if (n > 0 && pairs2 && cap > 0) {
    size_t tb = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, tb, a.as<uint32_t>(), b.as<uint32_t>(), (int)n, 0, 32, st);
    STOCS_CUDA(ctx, tmp.ensure(tb));
    cub::DeviceRadixSort::SortKeys(tmp.p, tb, a.as<uint32_t>(), b.as<uint32_t>(), (int)n, 0, 32, st);
    std::vector<uint32_t> h((size_t)n);
    STOCS_CUDA(ctx, cudaMemcpyAsync(h.data(), b.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    STOCS_CUDA(ctx, cudaStreamSynchronize(st));
    for (long long i = 0; i < n && i < cap; ++i) {
      pairs2[2 * i] = (int32_t)(h[i] >> 16);
      pairs2[2 * i + 1] = (int32_t)(h[i] & 0xffff);
    }
  }
  a.release(); b.release(); tmp.release();
  return STOCS_OK;
}

}  // extern "C"

// ---- test hook: the fp32 angle estimates of ppf_device.cuh beside the pinned evaluation -------------
namespace {
__global__ void angle_estimates_kernel(const float* __restrict__ y, const float* __restrict__ x, long long n,
                                       float* __restrict__ est, double* __restrict__ pinned, int* __restrict__ fast_floor,
                                       int* __restrict__ pinned_floor, unsigned char* __restrict__ below30_fast,
                                       unsigned char* __restrict__ below30_pinned) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float yy = y[i], xx = x[i];
  est[i] = atan2f(yy, xx) * 57.29577951308232f;
  const double p = stocsm::deg_atan2_ref(yy, xx);
  pinned[i] = p;
  fast_floor[i] = deg_atan2_floor(yy, xx);
  pinned_floor[i] = (int)p;
  // the 30-degree predicate on d = x (y unused): fast form and the pinned statement of src/stocs.cpp:428-436
  below30_fast[i] = internal_angle_below_30(xx) ? 1 : 0;
  float ang = stocsm::deg_acos_unqualified_ref(xx);
  const float other = 180.0f - ang;
  ang = (other < ang) ? other : ang;
  below30_pinned[i] = (ang < 30.0f) ? 1 : 0;
}
}  // namespace

extern "C" int stocs_b200_debug_angle_estimates(stocs_b200_ctx* ctx, const float* y, const float* x, int64_t n, float* est_deg,
                                                double* pinned_deg, int32_t* fast_floor, int32_t* pinned_floor,
                                                uint8_t* below30_fast, uint8_t* below30_pinned) {
  if (!ctx) return STOCS_E_ARG;
  if (n <= 0 || !y || !x || !est_deg || !pinned_deg || !fast_floor || !pinned_floor || !below30_fast || !below30_pinned)
    STOCS_FAIL(ctx, STOCS_E_ARG, "debug_angle_estimates: bad argument");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  DevBuf in, out;
  auto fail = [&](const char* what) { in.release(); out.release(); ctx->err = what; return STOCS_E_CUDA; };
  if (in.ensure((size_t)n * 8) != cudaSuccess || out.ensure((size_t)n * (4 + 8 + 4 + 4 + 1 + 1) + 64) != cudaSuccess) return fail("debug_angle_estimates: allocation failed");
  float* d_y = in.as<float>(); float* d_x = d_y + n;
  double* d_p = out.as<double>(); float* d_e = (float*)(d_p + n); int* d_ff = (int*)(d_e + n); int* d_pf = d_ff + n;
  unsigned char* d_bf = (unsigned char*)(d_pf + n); unsigned char* d_bp = d_bf + n;
  bool ok = cudaMemcpyAsync(d_y, y, (size_t)n * 4, cudaMemcpyHostToDevice, st) == cudaSuccess &&
            cudaMemcpyAsync(d_x, x, (size_t)n * 4, cudaMemcpyHostToDevice, st) == cudaSuccess;
  if (ok) angle_estimates_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_y, d_x, n, d_e, d_p, d_ff, d_pf, d_bf, d_bp);
  ok = ok && cudaMemcpyAsync(est_deg, d_e, (size_t)n * 4, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
       cudaMemcpyAsync(pinned_deg, d_p, (size_t)n * 8, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
       cudaMemcpyAsync(fast_floor, d_ff, (size_t)n * 4, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
       cudaMemcpyAsync(pinned_floor, d_pf, (size_t)n * 4, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
       cudaMemcpyAsync(below30_fast, d_bf, (size_t)n, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
       cudaMemcpyAsync(below30_pinned, d_bp, (size_t)n, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
       cudaStreamSynchronize(st) == cudaSuccess;
  if (!ok) return fail("debug_angle_estimates: CUDA call failed");
  in.release(); out.release();
  return STOCS_OK;
}
