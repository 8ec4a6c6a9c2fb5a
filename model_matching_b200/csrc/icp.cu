// icp.cu -- point-to-plane ICP refinement on the device (reference src/pose_clustering.cpp:123-141:
// pcl::IterativeClosestPointWithNormals, 5 iterations, max correspondence distance 0.035).
//
// Per iteration two launches, nothing returns to the host until the loop ends:
//   icp_pairs_kernel   one thread per source point: move the point by the previous step's matrix,
//                      exact nearest target point (target staged through shared memory in tiles;
//                      lowest index on equal squared distances), the pair's 29 binary64 terms,
//                      butterfly sum per warp, warps in order -> one partial row per 256 points;
//   icp_solve_kernel   one warp: partial rows summed in block order, 6x6 solve, step matrix,
//                      final = step * final.
// The summation order is fixed (stocs_icp_math.h), so the result is bit-identical to the oracle's.
// Memory traffic is negligible (segments are thousands of points); the launches are latency bound.
#include <cstring>

#include "stocs_ctx.h"
#include "stocs_icp_math.h"

using namespace stocsm;

namespace {

constexpr int kTile = 1024;

struct IcpState {       // device-resident loop state
  float step[16];       // matrix the next pairs kernel applies to the source
  float final_T[16];    // accumulated transform
  int n_pairs[16];      // correspondences per iteration
  double sum_d2[16];    // sum of squared pair distances per iteration
  int iterations;       // completed iterations
  int failed;           // 1: fewer than 3 pairs or singular system (loop stops, like PCL's "not converged")
};

__global__ void icp_init_kernel(IcpState* st) {
  const int t = threadIdx.x;
  if (t < 16) {
    const float v = (t % 5 == 0) ? 1.f : 0.f;
    st->step[t] = v; st->final_T[t] = v; st->n_pairs[t] = 0; st->sum_d2[t] = 0.0;
  }
  if (t == 0) { st->iterations = 0; st->failed = 0; }
}

__global__ void __launch_bounds__(kIcpBlock)
icp_pairs_kernel(float4* __restrict__ src, int n_src, const float4* __restrict__ tgt, const float4* __restrict__ tgt_n,
                 int n_tgt, double max_d2, const IcpState* __restrict__ st, double* __restrict__ partial,
                 int* __restrict__ nn_out) {
  __shared__ float4 tile[kTile];
  __shared__ double wsum[kIcpBlock / 32][kIcpTerms];
  if (st->failed) return;  // uniform: the loop has stopped
  const int i = blockIdx.x * kIcpBlock + threadIdx.x;
  const bool live = i < n_src;
  V3 s = v3(0, 0, 0);
  if (live) {
    const float4 p = src[i];
    s = xform_point(st->step, v3(p.x, p.y, p.z));
    src[i] = make_float4(s.x, s.y, s.z, p.w);
  }
  float best = 3.4e38f;
  int best_j = -1;
  for (int base = 0; base < n_tgt; base += kTile) {
    const int cnt = min(kTile, n_tgt - base);
    __syncthreads();
    for (int t = threadIdx.x; t < cnt; t += kIcpBlock) tile[t] = tgt[base + t];
    __syncthreads();
    if (live)
      for (int t = 0; t < cnt; ++t) {
        const float4 q = tile[t];
        const float d2 = icp_sqdist(s, v3(q.x, q.y, q.z));
        if (d2 < best) { best = d2; best_j = base + t; }
      }
  }
  double t[kIcpTerms];
#pragma unroll
  for (int k = 0; k < kIcpTerms; ++k) t[k] = 0.0;
  const bool paired = live && best_j >= 0 && !((double)best > max_d2);
  if (paired) {
    const float4 q = tgt[best_j], n = tgt_n[best_j];
    icp_pair_terms(s, v3(q.x, q.y, q.z), v3(n.x, n.y, n.z), best, t);
  }
  if (live && nn_out) nn_out[i] = paired ? best_j : -1;
#pragma unroll
  for (int k = 0; k < kIcpTerms; ++k) {
    double v = t[k];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v = v + __shfl_xor_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < kIcpTerms) {
    double acc = wsum[0][threadIdx.x];
    for (int w = 1; w < kIcpBlock / 32; ++w) acc = acc + wsum[w][threadIdx.x];
    partial[(size_t)blockIdx.x * kIcpTerms + threadIdx.x] = acc;
  }
}

__global__ void icp_solve_kernel(const double* __restrict__ partial, int nblocks, IcpState* st) {
  __shared__ double tot[kIcpTerms];
  if (st->failed) return;
  const int t = threadIdx.x;
  if (t < kIcpTerms) {
    double acc = partial[t];
    for (int b = 1; b < nblocks; ++b) acc = acc + partial[(size_t)b * kIcpTerms + t];
    tot[t] = acc;
  }
  __syncthreads();
  if (t == 0) {
    const int it = st->iterations;
    const int pairs = (int)tot[27];
    st->n_pairs[it] = pairs;
    st->sum_d2[it] = tot[28];
    double x[6];
    if (pairs < 3 || !icp_solve6(tot, tot + 21, x)) {
      st->failed = 1;
      for (int k = 0; k < 16; ++k) st->step[k] = (k % 5 == 0) ? 1.f : 0.f;
      return;
    }
    float m[16], f[16];
    icp_construct(x, m);
    mat4_mul(m, st->final_T, f);
    for (int k = 0; k < 16; ++k) { st->step[k] = m[k]; st->final_T[k] = f[k]; }
    st->iterations = it + 1;
  }
}

// apply the last step to the source (the aligned segment the reference leaves in segment_cloud)
__global__ void icp_apply_kernel(float4* __restrict__ src, int n_src, const IcpState* __restrict__ st) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_src) return;
  const float4 p = src[i];
  const V3 s = xform_point(st->step, v3(p.x, p.y, p.z));
  src[i] = make_float4(s.x, s.y, s.z, p.w);
}

}  // namespace

extern "C" int stocs_b200_icp_point_to_plane(stocs_b200_ctx* ctx, const float* src_pos3, int n_src,
                                             const float* tgt_pos3, const float* tgt_nrm3, int n_tgt,
                                             int max_iterations, float max_correspondence_distance,
                                             float* T16_out, float* aligned_pos3, int32_t* pairs_per_iteration,
                                             int32_t* iterations_done, int32_t* converged) {
  if (!ctx) return STOCS_E_ARG;
  if (!src_pos3 || !tgt_pos3 || !tgt_nrm3 || n_src <= 0 || n_tgt <= 0 || !T16_out)
    STOCS_FAIL(ctx, STOCS_E_ARG, "icp: bad argument");
  if (max_iterations < 1 || max_iterations > 16) STOCS_FAIL(ctx, STOCS_E_ARG, "icp: 1..16 iterations");
  if (!(max_correspondence_distance > 0)) STOCS_FAIL(ctx, STOCS_E_ARG, "icp: max_correspondence_distance must be positive");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  DevBuf &d_src = ctx->pool[POOL_ICP_SRC], &d_tgt = ctx->pool[POOL_ICP_TGT], &d_tn = ctx->pool[POOL_ICP_TN], &d_part = ctx->pool[POOL_ICP_PART], &d_state = ctx->pool[POOL_ICP_STATE];
  const int nblocks = (n_src + kIcpBlock - 1) / kIcpBlock;
  STOCS_CUDA(ctx, d_src.ensure((size_t)n_src * 16));
  STOCS_CUDA(ctx, d_tgt.ensure((size_t)n_tgt * 16));
  STOCS_CUDA(ctx, d_tn.ensure((size_t)n_tgt * 16));
  STOCS_CUDA(ctx, d_part.ensure((size_t)nblocks * kIcpTerms * 8));
  STOCS_CUDA(ctx, d_state.ensure(sizeof(IcpState)));
  std::vector<float4> h((size_t)(n_src > n_tgt ? n_src : n_tgt));
  auto pack = [&](const float* p3, int n, DevBuf& dst) -> cudaError_t {
    for (int i = 0; i < n; ++i) h[i] = make_float4(p3[3 * i], p3[3 * i + 1], p3[3 * i + 2], 0.f);
    cudaError_t e = cudaMemcpyAsync(dst.p, h.data(), (size_t)n * 16, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // h is reused
    return e;
  };
  STOCS_CUDA(ctx, pack(src_pos3, n_src, d_src));
  STOCS_CUDA(ctx, pack(tgt_pos3, n_tgt, d_tgt));
  STOCS_CUDA(ctx, pack(tgt_nrm3, n_tgt, d_tn));
  IcpState* ds = d_state.as<IcpState>();
  icp_init_kernel<<<1, 32, 0, st>>>(ds);
  const double max_d2 = (double)max_correspondence_distance * (double)max_correspondence_distance;
  for (int it = 0; it < max_iterations; ++it) {
    icp_pairs_kernel<<<nblocks, kIcpBlock, 0, st>>>(d_src.as<float4>(), n_src, d_tgt.as<float4>(), d_tn.as<float4>(), n_tgt,
                                                    max_d2, ds, d_part.as<double>(), nullptr);
    icp_solve_kernel<<<1, 32, 0, st>>>(d_part.as<double>(), nblocks, ds);
  }
  icp_apply_kernel<<<nblocks, kIcpBlock, 0, st>>>(d_src.as<float4>(), n_src, ds);
  STOCS_CUDA(ctx, cudaGetLastError());
  IcpState hs;
  STOCS_CUDA(ctx, cudaMemcpyAsync(&hs, ds, sizeof(hs), cudaMemcpyDeviceToHost, st));
  if (aligned_pos3) STOCS_CUDA(ctx, cudaMemcpyAsync(h.data(), d_src.p, (size_t)n_src * 16, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  if (aligned_pos3)
    for (int i = 0; i < n_src; ++i) { aligned_pos3[3 * i] = h[i].x; aligned_pos3[3 * i + 1] = h[i].y; aligned_pos3[3 * i + 2] = h[i].z; }
  memcpy(T16_out, hs.final_T, 64);
  if (pairs_per_iteration)
    for (int it = 0; it < max_iterations; ++it) pairs_per_iteration[it] = hs.n_pairs[it];
  if (iterations_done) *iterations_done = hs.iterations;
  if (converged) *converged = hs.failed ? 0 : 1;
  ctx->counters[CTR_SCORE_LAUNCHES] += 2 * max_iterations + 2;
  return STOCS_OK;
}
