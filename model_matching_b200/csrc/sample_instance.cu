// sample_instance.cu -- edge-aware ("instance") base sampling.
//
// Replaces stocs_estimator::sample_instance_base (reference src/stocs.cpp:559-751),
// prune_edge_pixels (:521-535) and rgbd::generate_segmentation_mask (src/rgbd.cpp:314-367).
// Bases are sequentially coupled in this mode (previous_segment decays the class prior
// permanently, segmentation_buffer caches earlier masks), so one launch = one base, one CTA of
// 32 warps; the parallelism is inside the base: per-point passes as in sample.cu, and the
// 8-connected flood fill over non-edge pixels as a level-synchronous BFS (claim = atomicOr on the
// mask word, frontier queues in global memory).  The reference caches masks as
// dbg/seg_mask_<n>.png and re-reads them; here they stay in device memory (lossless either way).
#include "sample_common.cuh"
#include "stocs_ctx.h"

using namespace stocsm;
using namespace stocs_sample;

PpfView stocs_ppf_view(const stocs_b200_ctx* ctx);

namespace {

struct InstArgs {
  const float4* __restrict__ spos4;
  float4* sattr;               // .w (class probability) is decayed in place
  const int2* __restrict__ spix;  // (row, col)
  int S;
  PpfView ppf;
  unsigned long long seed;
  int base_num;                // 1-based, also the RNG base number
  float dispersion;
  const uint8_t* __restrict__ edge;
  uint8_t* prev_mask;
  uint8_t* seg_buffer;
  uint8_t* cur_mask;           // scratch, H*W (multiple of 4)
  uint8_t* mask_store;         // 256 masks
  int* frontier;               // 2 * H*W
  int W, H;
  uint32_t* alive;             // ceil(S/32) words
  uint32_t* seg_alive;         // survivors right after the mask (the reference's `segment` output)
  int words;
  int* out_ids;
  float* out_inv;
  uint8_t* out_valid;
};

struct Shared {
  unsigned long long wsum[32];
  unsigned long long rem;
  int b[4];
  int pw;
  int maxdist_bits;
  int fcount[2];
};

// block-wide categorical draw over the alive points; returns the index or -1 (uniform)
__device__ int block_draw(const InstArgs& a, Shared& s, unsigned long long lsum, int draw_no, int t0, int t1) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  lsum = warp_sum_u64(lsum);
  if (lane == 0) s.wsum[w] = lsum;
  __syncthreads();
  if (tid == 0) {
    unsigned long long total = 0;
    for (int k = 0; k < 32; ++k) total += s.wsum[k];
    if (total == 0) {
      s.pw = -1;
    } else {
      unsigned long long r = mulhi_u64(draw_u64(a.seed, (uint32_t)a.base_num, (uint32_t)draw_no), total);
      int k = 0;
      while (k < 31 && r >= s.wsum[k]) { r -= s.wsum[k]; ++k; }
      s.pw = k;
      s.rem = r;
    }
  }
  __syncthreads();
  if (s.pw < 0) return -1;
  if (w == s.pw) {
    unsigned long long rem = s.rem;
    for (int t = t0; t < t1; ++t) {
      const int i = t * 32 + lane;
      unsigned long long wt = 0;
      if (i < a.S && ((a.alive[t] >> lane) & 1u)) wt = prob_weight(a.sattr[i].w);
      unsigned long long inc = wt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += up;
      }
      const unsigned long long tile_total = __shfl_sync(0xffffffffu, inc, 31);
      if (rem < tile_total) {
        const unsigned hit = __ballot_sync(0xffffffffu, inc > rem);
        if (lane == 0) s.b[draw_no] = t * 32 + (__ffs(hit) - 1);
        break;
      }
      rem -= tile_total;
    }
  }
  __syncthreads();
  return s.b[draw_no];
}

__device__ __forceinline__ float pixel_dist(int r0, int c0, int r1, int c1) {
  const int dr = r0 - r1, dc = c0 - c1;
  return (float)sqrt((double)(dr * dr) + (double)(dc * dc));  // std::sqrt(std::pow(.,2)+std::pow(.,2)) -> float
}

__device__ void fail_out(const InstArgs& a) {
  if (threadIdx.x == 0) {
    a.out_valid[0] = 0;
    for (int k = 0; k < 4; ++k) a.out_ids[k] = -1;
    a.out_inv[0] = 0.f; a.out_inv[1] = 0.f;
  }
}

__global__ void __launch_bounds__(1024) sample_instance_kernel(InstArgs a) {
  __shared__ Shared s;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int tiles = a.words, tpw = (tiles + 31) / 32;
  const int t0 = w * tpw, t1 = min(tiles, t0 + tpw);
  const int npix = a.W * a.H;

  // prior decay inside the previous segment (permanent), reset, prune_edge_pixels
  unsigned long long lsum = 0;
  for (int t = t0; t < t1; ++t) {
    const int i = t * 32 + lane;
    bool al = false;
    float cls = 0.f;
    if (i < a.S) {
      const int2 px = a.spix[i];
      const int pi = px.x * a.W + px.y;
      cls = a.sattr[i].w;
      if (a.prev_mask[pi]) { cls = a.dispersion * cls; a.sattr[i].w = cls; }
      al = (cls != 0.0f) && (a.edge[pi] != 0);  // edge probability (255-e)/255 == 1 <=> e == 0
    }
    const unsigned word = __ballot_sync(0xffffffffu, al);
    if (lane == 0) a.alive[t] = word;
    if (al) lsum += prob_weight(cls);
  }
  if (tid == 0) s.maxdist_bits = 0;
  const int b1 = block_draw(a, s, lsum, 0, t0, t1);
  if (b1 < 0) { fail_out(a); return; }
  const float4 p1 = a.spos4[b1], n1 = a.sattr[b1];
  const V3 pb0 = v3(p1.x, p1.y, p1.z), nb0 = v3(n1.x, n1.y, n1.z);
  const int2 px1 = a.spix[b1];

  // pass 1: PPF(b1, i) must be a key of the model map; radius of the surviving pixels
  float lmax = 0.f;
  for (int t = t0; t < t1; ++t) {
    const int i = t * 32 + lane;
    bool al = false;
    if (i < a.S && ((a.alive[t] >> lane) & 1u)) {
      const float4 p4 = a.spos4[i], n4 = a.sattr[i];
      const Ppf4 f = ppf_compute_dev(pb0, nb0, v3(p4.x, p4.y, p4.z), v3(n4.x, n4.y, n4.z), a.ppf.tr, a.ppf.rot);
      al = ppf_key_exists(a.ppf, f) && i != b1;
      if (al) {
        const int2 px = a.spix[i];
        const float d = pixel_dist(px1.x, px1.y, px.x, px.y);
        if (d > lmax) lmax = d;
      }
    }
    const unsigned word = __ballot_sync(0xffffffffu, al);
    if (lane == 0) a.alive[t] = word;
  }
  atomicMax(&s.maxdist_bits, __float_as_int(lmax));  // non-negative floats order as ints
  __syncthreads();
  const float max_distance = __int_as_float(s.maxdist_bits);

  // segmentation mask: cached mask of the segment b1's pixel already belongs to, else flood fill
  uint32_t* mask32 = reinterpret_cast<uint32_t*>(a.cur_mask);
  const int seg = a.seg_buffer[px1.x * a.W + px1.y];
  if (seg != 0) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(a.mask_store + (size_t)seg * npix);
    for (int k = tid; k < npix / 4; k += blockDim.x) mask32[k] = src[k];
    __syncthreads();
  } else {
    for (int k = tid; k < npix / 4; k += blockDim.x) mask32[k] = 0u;
    if (tid == 0) { s.fcount[0] = 1; s.fcount[1] = 0; a.frontier[0] = px1.x * a.W + px1.y; }
    __syncthreads();
    if (tid == 0) {
      const int p = px1.x * a.W + px1.y;
      atomicOr(&mask32[p >> 2], 0xffu << (8 * (p & 3)));
      a.seg_buffer[p] = (uint8_t)a.base_num;
    }
    __syncthreads();
    int cur = 0;
    while (true) {
      const int n = s.fcount[cur];
      if (n == 0) break;
      int* fin = a.frontier + (size_t)cur * npix;
      int* fout = a.frontier + (size_t)(1 - cur) * npix;
      for (int k = tid; k < n * 9; k += blockDim.x) {
        const int p = fin[k / 9], nb = k % 9;
        const int i = p / a.W + (nb / 3 - 1), j = p % a.W + (nb % 3 - 1);
        if (i < 0 || j < 0 || i >= a.H || j >= a.W) continue;
        const int q = i * a.W + j;
        if (a.edge[q] != 255) continue;                          // edge probability (255-e)/255 == 0 <=> e == 255
        if (!(pixel_dist(px1.x, px1.y, i, j) < max_distance)) continue;
        const uint32_t bit = 0xffu << (8 * (q & 3));
        const uint32_t old = atomicOr(&mask32[q >> 2], bit);
        if ((old & bit) == 0) {
          a.seg_buffer[q] = (uint8_t)a.base_num;
          fout[atomicAdd(&s.fcount[1 - cur], 1)] = q;
        }
      }
      __syncthreads();
      if (tid == 0) s.fcount[cur] = 0;
      cur = 1 - cur;
      __syncthreads();
    }
  }
  {  // cv::imwrite(seg_mask_<base_num>.png) + segmentation_mask.copyTo(previous_segment)
    uint32_t* store = reinterpret_cast<uint32_t*>(a.mask_store + (size_t)a.base_num * npix);
    uint32_t* prev = reinterpret_cast<uint32_t*>(a.prev_mask);
    for (int k = tid; k < npix / 4; k += blockDim.x) { const uint32_t v = mask32[k]; store[k] = v; prev[k] = v; }
  }
  __syncthreads();

  // keep only the points inside the mask
  lsum = 0;
  for (int t = t0; t < t1; ++t) {
    const int i = t * 32 + lane;
    bool al = false;
    float cls = 0.f;
    if (i < a.S && ((a.alive[t] >> lane) & 1u)) {
      const int2 px = a.spix[i];
      al = a.cur_mask[px.x * a.W + px.y] != 0;
      cls = a.sattr[i].w;
    }
    const unsigned word = __ballot_sync(0xffffffffu, al);
    if (lane == 0) { a.alive[t] = word; a.seg_alive[t] = word; }
    if (al) lsum += prob_weight(cls);
  }
  const int b2 = block_draw(a, s, lsum, 1, t0, t1);
  if (b2 < 0) { fail_out(a); return; }
  const float4 p2 = a.spos4[b2], n2 = a.sattr[b2];
  const V3 pb1 = v3(p2.x, p2.y, p2.z), nb1 = v3(n2.x, n2.y, n2.z);
  const V3 v_1 = normalized(sub(pb1, pb0));

  lsum = 0;
  for (int t = t0; t < t1; ++t) {
    const int i = t * 32 + lane;
    bool al = false;
    float cls = 0.f;
    if (i < a.S && ((a.alive[t] >> lane) & 1u)) {
      const float4 p4 = a.spos4[i], n4 = a.sattr[i];
      const V3 p = v3(p4.x, p4.y, p4.z);
      cls = n4.w;
      const Ppf4 f = ppf_compute_dev(pb1, nb1, p, v3(n4.x, n4.y, n4.z), a.ppf.tr, a.ppf.rot);
      al = ppf_key_exists(a.ppf, f) && i != b2 && !angle_too_small(v_1, p, pb0);
    }
    const unsigned word = __ballot_sync(0xffffffffu, al);
    if (lane == 0) a.alive[t] = word;
    if (al) lsum += prob_weight(cls);
  }
  const int b3 = block_draw(a, s, lsum, 2, t0, t1);
  if (b3 < 0) { fail_out(a); return; }
  const float4 p3 = a.spos4[b3], n3 = a.sattr[b3];
  const V3 pb2 = v3(p3.x, p3.y, p3.z), nb2 = v3(n3.x, n3.y, n3.z);
  const Plane pl = fit_plane(pb0, pb1, pb2);

  lsum = 0;
  for (int t = t0; t < t1; ++t) {
    const int i = t * 32 + lane;
    bool al = false;
    float cls = 0.f;
    if (i < a.S && ((a.alive[t] >> lane) & 1u)) {
      const float4 p4 = a.spos4[i], n4 = a.sattr[i];
      const V3 p = v3(p4.x, p4.y, p4.z);
      cls = n4.w;
      const Ppf4 f = ppf_compute_dev(pb2, nb2, p, v3(n4.x, n4.y, n4.z), a.ppf.tr, a.ppf.rot);
      al = ppf_key_exists(a.ppf, f) && i != b3 && !off_plane_or_too_close(pl, p, pb0, pb1, pb2);
    }
    const unsigned word = __ballot_sync(0xffffffffu, al);
    if (lane == 0) a.alive[t] = word;
    if (al) lsum += prob_weight(cls);
  }
  const int b4 = block_draw(a, s, lsum, 3, t0, t1);
  if (b4 < 0) { fail_out(a); return; }
  if (tid == 0) {
    const int ids[4] = {b1, b2, b3, b4};
    const float4 p4 = a.spos4[b4];
    const V3 b[4] = {pb0, pb1, pb2, v3(p4.x, p4.y, p4.z)};
    int best[4];
    float inv1, inv2;
    const bool ok = order_base(b, best, inv1, inv2);
    for (int k = 0; k < 4; ++k) a.out_ids[k] = ok ? ids[best[k]] : ids[k];
    a.out_inv[0] = inv1; a.out_inv[1] = inv2;
    a.out_valid[0] = ok ? 1 : 0;
  }
}

}  // namespace

extern "C" {

int stocs_b200_upload_edge_map(stocs_b200_ctx* ctx, const uint8_t* edge, int W, int H) {
  if (!ctx) return STOCS_E_ARG;
  if (!edge || W <= 0 || H <= 0 || ((long long)W * H) % 4 != 0) STOCS_FAIL(ctx, STOCS_E_ARG, "upload_edge_map: W*H must be a positive multiple of 4");
  cudaSetDevice(ctx->device);
  const size_t n = (size_t)W * H;
  STOCS_CUDA(ctx, ctx->d_edge.ensure(n));
  STOCS_CUDA(ctx, ctx->d_inst_state.ensure(n * 3));          // previous_segment | segmentation_buffer | current mask
  STOCS_CUDA(ctx, ctx->d_mask_store.ensure(n * 256));
  STOCS_CUDA(ctx, ctx->d_frontier.ensure(n * 2 * sizeof(int)));
  STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->d_edge.p, edge, n, cudaMemcpyHostToDevice, ctx->stream));
  STOCS_CUDA(ctx, cudaMemsetAsync(ctx->d_inst_state.p, 0, n * 3, ctx->stream));
  STOCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->img_w = W; ctx->img_h = H;
  return STOCS_OK;
}

}  // extern "C"

// One base of the stateful instance-mode sequence, enqueued on st: outputs go to DEVICE memory
// (d_ids 4 ints, d_inv 2 floats, d_valid 1 byte); mask and segment bits stay in ctx buffers.  No
// synchronisation: the sequential coupling between bases (prior decay, cached masks) lives in device
// state and is ordered by the stream, so a whole sequence can be enqueued back to back.
int stocs_launch_sample_instance(stocs_b200_ctx* ctx, uint64_t seed, int base_num, float dispersion, int* d_ids,
                                 float* d_inv, uint8_t* d_valid, cudaStream_t st) {
  if (ctx->S <= 0 || ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "sample_instance_base: upload_model and upload_scene first");
  if (ctx->img_w <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "sample_instance_base: upload_edge_map first");
  if (!ctx->has_pixels) STOCS_FAIL(ctx, STOCS_E_STATE, "sample_instance_base: upload_scene was called without pixel coordinates");
  if (ctx->pix_min[0] < 0 || ctx->pix_min[1] < 0 || ctx->pix_max[0] >= ctx->img_h || ctx->pix_max[1] >= ctx->img_w)
    STOCS_FAIL(ctx, STOCS_E_ARG, "sample_instance_base: scene pixel coordinates fall outside the edge map");
  if (base_num < 1 || base_num > 255) STOCS_FAIL(ctx, STOCS_E_ARG, "sample_instance_base: base_num must be 1..255");
  const size_t n = (size_t)ctx->img_w * ctx->img_h;
  InstArgs a;
  a.spos4 = ctx->d_spos4.as<float4>();
  a.sattr = ctx->d_sattr.as<float4>();
  a.spix = ctx->d_spix.as<int2>();
  a.S = ctx->S;
  a.ppf = stocs_ppf_view(ctx);
  a.seed = seed; a.base_num = base_num; a.dispersion = dispersion;
  // the prior decay rewrites weights in place as fl(dispersion * w): inside [0, w_max] only for a
  // dispersion in [0, 1], so any other value turns off the top-K pruning bound for this scene
  if (!(dispersion >= 0.f && dispersion <= 1.f)) ctx->prune_ok = false;
  a.edge = ctx->d_edge.as<uint8_t>();
  a.prev_mask = ctx->d_inst_state.as<uint8_t>();
  a.seg_buffer = a.prev_mask + n;
  a.cur_mask = a.prev_mask + 2 * n;
  a.mask_store = ctx->d_mask_store.as<uint8_t>();
  a.frontier = ctx->d_frontier.as<int>();
  a.W = ctx->img_w; a.H = ctx->img_h;
  a.words = (ctx->S + 31) / 32;
  STOCS_CUDA(ctx, ctx->d_work.ensure((size_t)a.words * 8));
  a.alive = ctx->d_work.as<uint32_t>();
  a.seg_alive = a.alive + a.words;
  STOCS_CUDA(ctx, cudaMemsetAsync(a.seg_alive, 0, (size_t)a.words * 4, st));
  a.out_ids = d_ids; a.out_inv = d_inv; a.out_valid = d_valid;
  sample_instance_kernel<<<1, 1024, 0, st>>>(a);
  STOCS_CUDA(ctx, cudaGetLastError());
  return STOCS_OK;
}

extern "C" {

int stocs_b200_sample_instance_base(stocs_b200_ctx* ctx, uint64_t seed, int base_num, float dispersion,
                                    int32_t* base_idx4, float* inv2, uint8_t* valid, uint8_t* mask_out,
                                    uint32_t* segment_bits) {
  if (!ctx) return STOCS_E_ARG;
  if (!base_idx4 || !inv2 || !valid) STOCS_FAIL(ctx, STOCS_E_ARG, "sample_instance_base: bad argument");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  int* d_ids = ctx->scratch()->inst_ids;
  float* d_inv = ctx->scratch()->inst_inv;
  uint8_t* d_valid = &ctx->scratch()->inst_valid;
  int rc = stocs_launch_sample_instance(ctx, seed, base_num, dispersion, d_ids, d_inv, d_valid, st);
  if (rc) return rc;
  const size_t n = (size_t)ctx->img_w * ctx->img_h;
  const int words = (ctx->S + 31) / 32;
  const uint8_t* cur_mask = ctx->d_inst_state.as<uint8_t>() + 2 * n;
  const uint32_t* seg_alive = ctx->d_work.as<uint32_t>() + words;
  STOCS_CUDA(ctx, cudaMemcpyAsync(base_idx4, d_ids, 16, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(inv2, d_inv, 8, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(valid, d_valid, 1, cudaMemcpyDeviceToHost, st));
  if (mask_out) STOCS_CUDA(ctx, cudaMemcpyAsync(mask_out, cur_mask, n, cudaMemcpyDeviceToHost, st));
  if (segment_bits) STOCS_CUDA(ctx, cudaMemcpyAsync(segment_bits, seg_alive, (size_t)words * 4, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  return STOCS_OK;
}

int stocs_b200_get_class_probability(stocs_b200_ctx* ctx, float* out) {
  if (!ctx || !out) return STOCS_E_ARG;
  if (ctx->S <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "no scene");
  cudaSetDevice(ctx->device);
  std::vector<float> tmp((size_t)ctx->S * 4);
  STOCS_CUDA(ctx, cudaMemcpyAsync(tmp.data(), ctx->d_sattr.p, (size_t)ctx->S * 16, cudaMemcpyDeviceToHost, ctx->stream));
  STOCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < ctx->S; ++i) out[i] = tmp[4 * (size_t)i + 3];
  return STOCS_OK;
}

// replica maintenance for multi-GPU runs: overwrite the per-point class probability (the w component
// of the scene attribute records) with values read from another context
int stocs_b200_set_class_probability(stocs_b200_ctx* ctx, const float* cls) {
  if (!ctx || !cls) return STOCS_E_ARG;
  if (ctx->S <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "no scene");
  cudaSetDevice(ctx->device);
  ctx->prune_ok = false;   // until the new weights are in place and bounded
  STOCS_CUDA(ctx, cudaMemcpy2DAsync(ctx->d_sattr.as<char>() + 12, 16, cls, 4, 4, (size_t)ctx->S, cudaMemcpyHostToDevice, ctx->stream));
  STOCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  stocs_set_weight_bound(ctx, cls, ctx->S);
  return STOCS_OK;
}

}  // extern "C"
