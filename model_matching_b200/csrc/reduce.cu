// reduce.cu -- best-pose argmax and top-K candidates over the LCP array.
//
// Replaces the argmax loop of stocs_estimator::compute_best_transform (reference
// src/stocs.cpp:987-1001: FIRST strict maximum wins, index -1 when every score is 0) and produces
// the K best candidates that feed clustering::greedy_clustering (src/pose_clustering.cpp:79-122).
// Keys are (ordered lcp bits << 32) | ~index, so a larger key is a larger score or, at equal score,
// a smaller index; key 0 is "no entry" (the low word of a real key is never 0, indices being < 2^32 - 1).  Each warp keeps a sorted top-32 across its lanes (lane j = j-th best) and
// inserts with one ballot + shuffle per surviving key; a single-warp kernel merges the per-warp
// lists.  Memory traffic: one read of the LCP array.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>

#include "stocs_ctx.h"

namespace {

__device__ __forceinline__ void warp_insert(unsigned long long& mine, unsigned long long key, int lane) {
  // list is sorted descending across lanes; insert key, drop the smallest
  const unsigned ge = __ballot_sync(0xffffffffu, mine >= key);  // lanes that stay in front of key
  const int pos = __popc(ge);                                   // insertion position
  const unsigned long long up = __shfl_up_sync(0xffffffffu, mine, 1);
  if (lane == pos) mine = key;
  else if (lane > pos) mine = up;
}

// Order-preserving map of binary32 onto uint32 (sign bit flipped for positives, all bits for
// negatives), -0.0 folded onto +0.0: the clustering filter `lcp > threshold` admits lcp <= 0 when the
// threshold is negative, and its `>` holds -0.0 and +0.0 equal, so the index must break that tie.
__device__ __forceinline__ unsigned ordered_bits(float v) {
  const unsigned u = __float_as_uint(v == 0.f ? 0.f : v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_lcp(unsigned long long key) {
  const unsigned o = (unsigned)(key >> 32);
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
__device__ __forceinline__ unsigned long long make_key(float v, unsigned long long idx) {
  return ((unsigned long long)ordered_bits(v) << 32) | (0xffffffffull - (idx & 0xffffffffull));
}

// offer one key per lane to the warp's sorted list
__device__ __forceinline__ void warp_offer(unsigned long long& mine, unsigned long long key, int lane) {
  const unsigned long long kth = __shfl_sync(0xffffffffu, mine, 31);
  unsigned pass = __ballot_sync(0xffffffffu, key > kth);
  while (pass) {
    const int b = __ffs(pass) - 1;
    const unsigned long long k = __shfl_sync(0xffffffffu, key, b);
    const unsigned long long cur_kth = __shfl_sync(0xffffffffu, mine, 31);
    if (k > cur_kth) warp_insert(mine, k, lane);
    pass &= pass - 1;
  }
}

// Merge two lists that are BOTH sorted descending across the lanes (lane j = j-th best) into the top 32
// of their union, sorted: max(a[j], b[31-j]) is a bitonic sequence that holds exactly those 32 keys,
// and five compare-exchange stages sort it.  ~60 instructions, against up to 32 dependent insertions
// with warp_offer (the final merge kernel took 40 us per step with those: it sits on the critical
// path of every step, 10 % of a step when 10^6 hypotheses are sharded over 8 GPUs).
__device__ __forceinline__ unsigned long long shfl64(unsigned long long v, int src) {
  const unsigned lo = __shfl_sync(0xffffffffu, (unsigned)v, src), hi = __shfl_sync(0xffffffffu, (unsigned)(v >> 32), src);
  return ((unsigned long long)hi << 32) | lo;
}
__device__ __forceinline__ void warp_merge_sorted(unsigned long long& mine, unsigned long long other, int lane) {
  const unsigned long long rev = shfl64(other, 31 - lane);
  unsigned long long m = mine > rev ? mine : rev;
#pragma unroll
  for (int k = 16; k >= 1; k >>= 1) {
    const unsigned long long p = shfl64(m, lane ^ k);
    const bool keep_max = (lane & k) == 0;      // descending: the lower lane of a pair keeps the larger key
    m = keep_max ? (m > p ? m : p) : (m < p ? m : p);
  }
  mine = m;
}

// ONE launch: every CTA reduces its strided share of the LCP array to a sorted top-32 list (per-warp
// lists with ballot insertion, merged by warp 0); the CTA that finishes LAST (threadfence + atomic
// ticket) merges the per-CTA lists -- each of its 8 warps folds a strided share with the bitonic merge,
// then a 3-round tournament -- and writes the K winners, also packed as 64-byte records {lcp, inliers,
// global index, rows 0..2 of the transform} when rec_out != NULL (the unit of the multi-GPU all-gather,
// comm.cu).  Two launches with insertion merges took 55 us per step at 10^6 hypotheses, this one 13 us.
__global__ void __launch_bounds__(256) topk_kernel(const float* __restrict__ lcp, long long H, unsigned long long* __restrict__ lists,
                                                   unsigned* __restrict__ ticket, int K, long long index_offset,
                                                   long long* __restrict__ out_idx, float* __restrict__ out_lcp,
                                                   const float* __restrict__ T16, const int* __restrict__ inl,
                                                   stocs_b200_record* __restrict__ rec_out, const long long* __restrict__ H_dev) {
  if (H_dev) H = *H_dev;   // the online pipeline keeps its count on the device
  __shared__ unsigned long long s_keys[8 * 32];
  __shared__ bool s_last;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long warp = (long long)blockIdx.x * 8 + w;
  const long long nwarps = (long long)gridDim.x * 8;
  unsigned long long mine = 0ull;  // key 0 == "empty" (lcp 0 never qualifies: strict > 0)
  for (long long base = warp * 32; base < H; base += nwarps * 32) {
    const long long i = base + lane;
    const float v = (i < H) ? lcp[i] : 0.f;
    warp_offer(mine, (v > 0.f) ? make_key(v, (unsigned long long)i) : 0ull, lane);
  }
  s_keys[w * 32 + lane] = mine;
  __syncthreads();
  if (w == 0) {
    for (int k = 1; k < 8; ++k) warp_merge_sorted(mine, s_keys[k * 32 + lane], lane);
    lists[(long long)blockIdx.x * 32 + lane] = mine;
    __threadfence();
    if (lane == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // ---- last CTA: merge the gridDim.x sorted lists
  mine = 0ull;
  for (long long l = w; l < (long long)gridDim.x; l += 8)
    warp_merge_sorted(mine, __ldcg(lists + l * 32 + lane), lane);   // written by other CTAs: bypass L1
  s_keys[w * 32 + lane] = mine;
  __syncthreads();
  for (int stride = 1; stride < 8; stride <<= 1) {
    if ((w & (2 * stride - 1)) == 0) {
      warp_merge_sorted(mine, s_keys[(w + stride) * 32 + lane], lane);
      s_keys[w * 32 + lane] = mine;
    }
    __syncthreads();
  }
  if (w != 0) return;
  if (lane == 0) *ticket = 0u;      // ready for the next launch (launches on one context are stream-ordered)
  if (lane < K) {
    const long long local = (long long)(0xffffffffull - (mine & 0xffffffffull));
    if (out_idx) {
      if (mine == 0ull) { out_idx[lane] = -1; out_lcp[lane] = 0.f; }
      else {
        out_idx[lane] = local + index_offset;
        out_lcp[lane] = key_lcp(mine);
      }
    }
    if (rec_out) {
      stocs_b200_record r;
      r.lcp = 0.f; r.inliers = 0; r.index = -1;
#pragma unroll
      for (int k = 0; k < 12; ++k) r.T[k] = 0.f;
      if (mine != 0ull) {
        r.lcp = key_lcp(mine);
        r.inliers = inl ? inl[local] : 0;
        r.index = local + index_offset;
        const float* t = T16 + 16 * local;   // column-major 4x4 -> rows 0..2, row-major
#pragma unroll
        for (int rr = 0; rr < 3; ++rr)
#pragma unroll
          for (int c = 0; c < 4; ++c) r.T[rr * 4 + c] = t[c * 4 + rr];
      }
      rec_out[lane] = r;
    }
  }
}

// key of every entry i < H: make_key(lcp[i], i) when lcp[i] > threshold (and > 0 with positive_only,
// and ok[i] != 0 with ok), 0 otherwise.  The threshold is thr, or thr * *thr_scale computed here when
// thr_scale is given (a factor times a best score that lives on the device).  H_dev: entries at or
// beyond the device count get key 0.
__global__ void above_keys_kernel(const float* __restrict__ lcp, long long H, float thr, const float* __restrict__ thr_scale,
                                  bool positive_only, const uint8_t* __restrict__ ok, const long long* __restrict__ H_dev,
                                  unsigned long long* __restrict__ keys) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H) return;
  if (thr_scale) thr = thr * *thr_scale;
  const bool in = (!H_dev || i < *H_dev) && (!ok || ok[i]);
  const float v = in ? lcp[i] : 0.f;
  keys[i] = (in && v > thr && (!positive_only || v > 0.f)) ? make_key(v, (unsigned long long)i) : 0ull;
}
struct NonZero { __device__ bool operator()(unsigned long long k) const { return k != 0ull; } };
__global__ void unpack_keys_kernel(const unsigned long long* __restrict__ keys, long long n, long long* __restrict__ idx,
                                   float* __restrict__ val) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  idx[i] = (long long)(0xffffffffull - (keys[i] & 0xffffffffull));
  val[i] = key_lcp(keys[i]);
}

}  // namespace

// All hypotheses with lcp > threshold, ordered by (lcp descending, index ascending): the filter +
// sort that opens clustering::greedy_clustering (reference src/pose_clustering.cpp:93-101).
extern "C" int stocs_b200_select_above(stocs_b200_ctx* ctx, const float* lcp, int64_t H, float threshold,
                                       int64_t* index_out, float* lcp_out, int64_t cap, int64_t* n_out) {
  if (!ctx) return STOCS_E_ARG;
  if (H < 0 || H >= (1ll << 31) || !n_out || cap < 0) STOCS_FAIL(ctx, STOCS_E_ARG, "select_above: bad argument");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  *n_out = 0;
  if (H == 0) return STOCS_OK;
  const float* d_src = nullptr;
  if (lcp) {
    STOCS_CUDA(ctx, ctx->d_lcp.ensure((size_t)H * 4));
    STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->d_lcp.p, lcp, (size_t)H * 4, cudaMemcpyHostToDevice, st));
    ctx->last_H = H;
    ctx->top_valid = false;
  } else if (ctx->last_H != H || !ctx->d_lcp.p) {
    STOCS_FAIL(ctx, STOCS_E_STATE, "select_above: no resident lcp array of that size");
  }
  d_src = ctx->d_lcp.as<float>();
  DevBuf ka, kb, tmp, cnt, oi, ov;
  auto cleanup = [&]() { ka.release(); kb.release(); tmp.release(); cnt.release(); oi.release(); ov.release(); };
#define SA(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) { ctx->err = std::string(#call) + ": " + cudaGetErrorString(_e); cleanup(); return STOCS_E_CUDA; } } while (0)
  SA(ka.ensure((size_t)H * 8)); SA(kb.ensure((size_t)H * 8)); SA(cnt.ensure(16));
  above_keys_kernel<<<(unsigned)((H + 255) / 256), 256, 0, st>>>(d_src, H, threshold, nullptr, true, nullptr, nullptr,
                                                                  ka.as<unsigned long long>());
  size_t tb = 0, tb2 = 0;
  cub::DeviceSelect::If(nullptr, tb, ka.as<unsigned long long>(), kb.as<unsigned long long>(), cnt.as<int>(), (int)H, NonZero(), st);
  cub::DeviceRadixSort::SortKeysDescending(nullptr, tb2, kb.as<unsigned long long>(), ka.as<unsigned long long>(), (int)H, 0, 64, st);
  SA(tmp.ensure(tb > tb2 ? tb : tb2));
  cub::DeviceSelect::If(tmp.p, tb, ka.as<unsigned long long>(), kb.as<unsigned long long>(), cnt.as<int>(), (int)H, NonZero(), st);
  int n = 0;
  SA(cudaMemcpyAsync(&n, cnt.p, 4, cudaMemcpyDeviceToHost, st));
  SA(cudaStreamSynchronize(st));
  *n_out = n;
  if (n > cap) { cleanup(); STOCS_FAIL(ctx, STOCS_E_CAPACITY, "select_above: capacity too small"); }
  if (n > 0) {
    if (!index_out || !lcp_out) { cleanup(); STOCS_FAIL(ctx, STOCS_E_ARG, "select_above: output pointer is NULL"); }
    cub::DeviceRadixSort::SortKeysDescending(tmp.p, tb2, kb.as<unsigned long long>(), ka.as<unsigned long long>(), n, 0, 64, st);
    SA(oi.ensure((size_t)n * 8)); SA(ov.ensure((size_t)n * 4));
    unpack_keys_kernel<<<(n + 255) / 256, 256, 0, st>>>(ka.as<unsigned long long>(), n, oi.as<long long>(), ov.as<float>());
    SA(cudaMemcpyAsync(index_out, oi.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    SA(cudaMemcpyAsync(lcp_out, ov.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    SA(cudaStreamSynchronize(st));
  }
#undef SA
  cleanup();
  return STOCS_OK;
}

int stocs_launch_topk(stocs_b200_ctx* ctx, const float* d_lcp, int64_t H, int K, int64_t index_offset,
                      cudaStream_t st, const TopkRequest& rq) {
  if (K < 1 || K > 32) STOCS_FAIL(ctx, STOCS_E_ARG, "reduce_best: K must be in 1..32");
  if (H >= (1ll << 32)) STOCS_FAIL(ctx, STOCS_E_ARG, "reduce_best: H must be < 2^32");
  int blocks = ctx->num_sms * 2;
  long long need = ((rq.d_H && rq.grid_hint > 0 && rq.grid_hint < H ? rq.grid_hint : H) + 2047) / 2048;   // at least 256 keys per warp: fewer, longer lists for the merge
  if (need < 1) need = 1;
  if (blocks > need) blocks = (int)need;
  // per-stream scratch: launches on the context stream and on its second stream (the host-buffer
  // calls overlap their result copies with the reduction) must not share lists or ticket
  const int which = (st == ctx->aux_stream) ? 1 : 0;
  DevBuf& lists = which ? ctx->pool[POOL_TOPK_LISTS_AUX] : ctx->d_work;
  STOCS_CUDA(ctx, lists.ensure((size_t)blocks * 32 * 8));
  unsigned* ticket = &ctx->scratch()->topk_ticket[which];   // zero at creation, reset by the last CTA
  topk_kernel<<<blocks, 256, 0, st>>>(d_lcp, H, lists.as<unsigned long long>(), ticket, K, index_offset,
                                      (long long*)rq.idx, rq.val, rq.T16, rq.inl, rq.rec, rq.d_H);
  STOCS_CUDA(ctx, cudaGetLastError());
  return STOCS_OK;
}

// The filter + order of clustering::greedy_clustering over a device list, without a host round trip:
// keys[0..H) = make_key of every entry with (ok[i] and) lcp[i] > thr * *thr_scale (or > thr), sorted
// descending into keys_out, non-candidates (key 0) last.  tmp / tmp_bytes: cub scratch (query with
// tmp == NULL: *tmp_bytes is set and nothing is enqueued).
int stocs_enqueue_cluster_keys(stocs_b200_ctx* ctx, const float* d_lcp, int64_t H, float thr, const float* d_thr_scale,
                               const uint8_t* d_ok, const long long* d_H, unsigned long long* keys,
                               unsigned long long* keys_out, void* tmp, size_t* tmp_bytes, cudaStream_t st) {
  if (!tmp) {
    STOCS_CUDA(ctx, cub::DeviceRadixSort::SortKeysDescending(nullptr, *tmp_bytes, keys, keys_out, (int)H, 0, 64, st));
    return STOCS_OK;
  }
  if (H == 0) return STOCS_OK;
  above_keys_kernel<<<(unsigned)((H + 255) / 256), 256, 0, st>>>(d_lcp, H, thr, d_thr_scale, false, d_ok, d_H, keys);
  STOCS_CUDA(ctx, cudaGetLastError());
  STOCS_CUDA(ctx, cub::DeviceRadixSort::SortKeysDescending(tmp, *tmp_bytes, keys, keys_out, (int)H, 0, 64, st));
  return STOCS_OK;
}
