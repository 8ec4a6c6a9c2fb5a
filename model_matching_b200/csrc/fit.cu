// fit.cu -- rigid transform per (base, congruent quad) and the fused online pipeline.
//
// fit_kernel replaces ComputeRigidTransformation (reference src/stocs.cpp:270-361) and
// stocs_estimator::get_rigid_transform_from_congruent_pair (:871-941): Gram-Schmidt frames on
// the first three correspondences, R = Fp^T Fq, the reference's (R*R).diagonal() orthogonality
// test, T = [R | c1 - R c2], and the un-centred pose with translation
// c1 + c_scene - R (c2 + c_model).  One thread per item; deviations D1 (degenerate input is
// rejected) and D4 (no SVD) as documented in oracle/stocs_oracle.cpp and DESIGN.md.
//
// stocs_b200_run_pipeline chains sample -> congruent -> select -> fit -> score -> reduce on the
// device (run_stocs_estimation, src/stocs_match_one_object.cpp:79-165).
#include <vector>

#include "stocs_ctx.h"

using namespace stocsm;

int stocs_launch_sample(stocs_b200_ctx* ctx, uint64_t seed, uint32_t first_base_no, int n_bases, int* d_ids,
                        float* d_inv, uint8_t* d_valid, cudaStream_t st);
int stocs_congruent_enqueue(stocs_b200_ctx* ctx, int n_bases, const int* d_base_idx4, const float* d_inv2,
                            const uint8_t* d_valid, StocsPipeState* d_state, long long* d_quad_off, cudaStream_t st);  // congruent.cu
bool stocs_congruent_grow(stocs_b200_ctx* ctx, const StocsPipeState& s);

namespace {

__device__ __forceinline__ V3 ld3(const float4* p, int i) { const float4 v = p[i]; return v3(v.x, v.y, v.z); }
__device__ __forceinline__ float comp(const V3& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : v.z); }

__device__ __forceinline__ bool make_frame(V3 a0, V3 a1, V3 a2, V3 f[3]) {
  V3 v1 = sub(a1, a0);
  if (sqnorm(v1) == 0) return false;
  v1 = normalized(v1);
  const V3 d = sub(a2, a0);
  V3 v2 = sub(d, scale(v1, dot(d, v1)));
  if (sqnorm(v2) == 0) return false;
  v2 = normalized(v2);
  f[0] = v1; f[1] = v2; f[2] = cross(v1, v2);
  return true;
}

// item t: base ids base_idx4[4*bmap(t)..], quad quads4[4*qmap(t)..]
struct FitArgs {
  const float4* __restrict__ spos4;
  const float4* __restrict__ mpos4;
  const int* __restrict__ base_idx4;
  const int* __restrict__ quads4;
  const int* __restrict__ item_base;   // optional: item -> base row (NULL: identity)
  const long long* __restrict__ item_quad;  // optional: item -> quad row (NULL: identity)
  float* __restrict__ Tc;
  float* __restrict__ Tw;
  uint8_t* __restrict__ ok;
  long long n;
  const long long* __restrict__ n_dev;  // optional: the item count lives on the device (n is then ignored)
  float cs[3], cm[3];
  int S, M;
};

__global__ void fit_kernel(FitArgs a) {
  const long long n = a.n_dev ? *a.n_dev : a.n;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
  const int* bid = a.base_idx4 + 4 * (size_t)(a.item_base ? a.item_base[t] : t);
  const int* qd = a.quads4 + 4 * (size_t)(a.item_quad ? a.item_quad[t] : t);
  float* Tc = a.Tc + 16 * (size_t)t;
  float* Tw = a.Tw ? a.Tw + 16 * (size_t)t : nullptr;
  bool good = true;
  for (int k = 0; k < 3; ++k) good = good && bid[k] >= 0 && bid[k] < a.S && qd[k] >= 0 && qd[k] < a.M;
  float R[3][3];
  V3 c1 = v3(0, 0, 0), c2 = v3(0, 0, 0);
  if (good) {
    const V3 p0 = ld3(a.spos4, bid[0]), p1 = ld3(a.spos4, bid[1]), p2 = ld3(a.spos4, bid[2]);
    const V3 q0 = ld3(a.mpos4, qd[0]), q1 = ld3(a.mpos4, qd[1]), q2 = ld3(a.mpos4, qd[2]);
    c1 = divs(add(add(p0, p1), p2), 3.0f);
    c2 = divs(add(add(q0, q1), q2), 3.0f);
    V3 fp[3], fq[3];
    good = make_frame(p0, p1, p2, fp) && make_frame(q0, q1, q2, fq);
    if (good) {
      for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
          R[i][j] = sum3(comp(fp[0], i) * comp(fq[0], j), comp(fp[1], i) * comp(fq[1], j), comp(fp[2], i) * comp(fq[2], j));
      for (int i = 0; i < 3; ++i) {
        const float rr = sum3(R[i][0] * R[0][i], R[i][1] * R[1][i], R[i][2] * R[2][i]);
        if (rr - 1.0f > 1e-6f) good = false;
        if (rr != rr) good = false;
      }
    }
  }
  if (!good) {
    // rejected items carry NaN so that, if they are scored anyway, they can never win
    const float qnan = __int_as_float(0x7fc00000);
    for (int k = 0; k < 16; ++k) { Tc[k] = qnan; if (Tw) Tw[k] = qnan; }
    a.ok[t] = 0;
    continue;
  }
  const V3 nc2 = v3(-c2.x, -c2.y, -c2.z);
  const float c1a[3] = {c1.x, c1.y, c1.z};
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) { Tc[j * 4 + i] = R[i][j]; if (Tw) Tw[j * 4 + i] = R[i][j]; }
    Tc[12 + i] = c1a[i] + sum3(R[i][0] * nc2.x, R[i][1] * nc2.y, R[i][2] * nc2.z);
  }
  Tc[3] = Tc[7] = Tc[11] = 0.f; Tc[15] = 1.f;
  if (Tw) {
    const V3 sa = add(c1, v3(a.cs[0], a.cs[1], a.cs[2]));
    const V3 sb = add(c2, v3(a.cm[0], a.cm[1], a.cm[2]));
    const float saa[3] = {sa.x, sa.y, sa.z};
    for (int i = 0; i < 3; ++i) Tw[12 + i] = saa[i] - sum3(R[i][0] * sb.x, R[i][1] * sb.y, R[i][2] * sb.z);
    Tw[3] = Tw[7] = Tw[11] = 0.f; Tw[15] = 1.f;
  }
  a.ok[t] = 1;
  }
}

// item offsets of the pipeline from the per-base quad offsets: min(cnt, max_sets) transforms per base
// (one block; the total goes to the state record)
__global__ void __launch_bounds__(256) pipe_item_offsets_kernel(const long long* __restrict__ quad_off, int n_bases, int max_sets,
                                                                 long long* __restrict__ item_off, StocsPipeState* __restrict__ stt) {
  __shared__ unsigned long long s_buf[256];
  const int j = threadIdx.x;
  const int per = (n_bases + 255) / 256;
  const int b0 = min(n_bases, j * per), b1 = min(n_bases, b0 + per);
  unsigned long long loc = 0;
  for (int b = b0; b < b1; ++b) { const long long c = quad_off[b + 1] - quad_off[b]; loc += (unsigned long long)(c < max_sets ? c : max_sets); }
  // exclusive scan of the 256 partial sums
  s_buf[j] = loc;
  __syncthreads();
  for (int o = 1; o < 256; o <<= 1) {
    const unsigned long long up = (j >= o) ? s_buf[j - o] : 0ull;
    __syncthreads();
    s_buf[j] += up;
    __syncthreads();
  }
  unsigned long long off = s_buf[j] - loc;
  for (int b = b0; b < b1; ++b) {
    item_off[b] = (long long)off;
    const long long c = quad_off[b + 1] - quad_off[b];
    off += (unsigned long long)(c < max_sets ? c : max_sets);
  }
  if (j == 255) { item_off[n_bases] = (long long)s_buf[255]; stt->n_items = (long long)s_buf[255]; }
}

// closes a pipeline run (one block): the best hypothesis -- first strict maximum of the LCP array, as
// reduce.cu orders its keys: (lcp bits, lower index first), lcp > 0 only; taken from best_idx/best_val
// instead when the caller ran the general top-K reduction (lcp == NULL) --, the transforms that passed
// the fit, the winner's rank among them (the index the reference's transform list gives it), its
// base's rank among the valid bases, its two poses
__global__ void __launch_bounds__(1024) pipe_finalize_kernel(const float* __restrict__ lcp, const uint8_t* __restrict__ ok,
                                                              const uint8_t* __restrict__ valid, int n_bases,
                                                              const int* __restrict__ item_base, const long long* __restrict__ best_idx,
                                                              const float* __restrict__ best_val, const float* __restrict__ Tc,
                                                              const float* __restrict__ Tw, StocsPipeState* __restrict__ stt) {
  __shared__ unsigned long long s_key[32];
  __shared__ long long s_a[32], s_b[32];
  __shared__ int s_c[32], s_d[32];
  __shared__ long long s_bi;
  __shared__ float s_bv;
  const int j = threadIdx.x, lane = j & 31, w = j >> 5;
  const long long n = stt->n_items;
  if (lcp) {
    unsigned long long key = 0ull;
    for (long long i = j; i < n; i += 1024) {
      const float v = lcp[i];
      const unsigned long long k = (v > 0.f) ? (((unsigned long long)__float_as_uint(v) << 32) | (0xffffffffull - (unsigned long long)i)) : 0ull;
      key = k > key ? k : key;
    }
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o); key = other > key ? other : key; }
    if (lane == 0) s_key[w] = key;
    __syncthreads();
    if (j == 0) {
      for (int k = 1; k < 32; ++k) key = s_key[k] > key ? s_key[k] : key;
      s_bi = key ? (long long)(0xffffffffull - (key & 0xffffffffull)) : -1ll;
      s_bv = key ? __uint_as_float((unsigned)(key >> 32)) : 0.f;
    }
  } else if (j == 0) {
    s_bi = best_idx[0];
    s_bv = best_val[0];
  }
  __syncthreads();
  const long long bi = s_bi;
  long long n_ok = 0, before = 0;
  for (long long i = j; i < n; i += 1024) { const int o = ok[i] ? 1 : 0; n_ok += o; if (i < bi) before += o; }
  const int bb = (bi >= 0) ? item_base[bi] : -1;
  int n_valid = 0, valid_before = 0;
  for (int b = j; b < n_bases; b += 1024) { const int o = valid[b] ? 1 : 0; n_valid += o; if (b < bb) valid_before += o; }
  for (int o = 16; o > 0; o >>= 1) {
    n_ok += __shfl_xor_sync(0xffffffffu, n_ok, o); before += __shfl_xor_sync(0xffffffffu, before, o);
    n_valid += __shfl_xor_sync(0xffffffffu, n_valid, o); valid_before += __shfl_xor_sync(0xffffffffu, valid_before, o);
  }
  if (lane == 0) { s_a[w] = n_ok; s_b[w] = before; s_c[w] = n_valid; s_d[w] = valid_before; }
  __syncthreads();
  if (j == 0) {
    for (int k = 1; k < 32; ++k) { n_ok += s_a[k]; before += s_b[k]; n_valid += s_c[k]; valid_before += s_d[k]; }
    stt->n_ok = n_ok;
    stt->n_valid = n_valid;
    stt->best_item = bi;
    stt->rank_of_best = (bi >= 0) ? before : -1;
    stt->best_base = (bi >= 0) ? valid_before : -1;
    stt->best_lcp = s_bv;
  }
  if (j < 16) {
    stt->best_Tc[j] = (bi >= 0) ? Tc[16 * bi + j] : 0.f;
    stt->best_Tw[j] = (bi >= 0) ? Tw[16 * bi + j] : 0.f;
  }
}

// item list of the pipeline: for base b with cnt quads, take all when cnt < max_sets, else
// max_sets quads spread evenly over the (sorted) list: index floor(k * cnt / max_sets).
__global__ void select_items_kernel(const long long* __restrict__ quad_off, const long long* __restrict__ item_off,
                                    int n_bases, int max_sets, int* __restrict__ item_base,
                                    long long* __restrict__ item_quad) {
  const int b = blockIdx.x;
  const long long q0 = quad_off[b], cnt = quad_off[b + 1] - q0;
  const long long o = item_off[b];
  const long long take = cnt < max_sets ? cnt : max_sets;
  for (long long k = threadIdx.x; k < take; k += blockDim.x) {
    const long long src = (cnt < max_sets) ? k : (k * cnt) / max_sets;
    item_base[o + k] = b;
    item_quad[o + k] = q0 + src;
  }
}

}  // namespace

static void fill_fit_args(stocs_b200_ctx* ctx, FitArgs& a) {
  a.spos4 = ctx->d_spos4.as<float4>();
  a.mpos4 = ctx->d_mpos4.as<float4>();
  for (int k = 0; k < 3; ++k) { a.cs[k] = ctx->cs[k]; a.cm[k] = ctx->cm[k]; }
  a.S = ctx->S; a.M = ctx->M;
  a.item_base = nullptr; a.item_quad = nullptr; a.n_dev = nullptr;
}

extern "C" int stocs_b200_fit_transforms(stocs_b200_ctx* ctx, int64_t n, const int32_t* base_idx4, const int32_t* quads4,
                                         float* T_centred16, float* T_world16, uint8_t* ok) {
  if (!ctx) return STOCS_E_ARG;
  if (ctx->S <= 0 || ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "fit_transforms: upload_model and upload_scene first");
  if (n < 0 || (n > 0 && (!base_idx4 || !quads4 || !T_centred16 || !ok))) STOCS_FAIL(ctx, STOCS_E_ARG, "fit_transforms: bad argument");
  if (n == 0) return STOCS_OK;
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  STOCS_CUDA(ctx, ctx->d_tmp.ensure((size_t)n * 32));
  STOCS_CUDA(ctx, ctx->d_tmp2.ensure((size_t)n * (128 + 1) + 64));
  int* d_b = ctx->d_tmp.as<int>();
  int* d_q = d_b + 4 * (size_t)n;
  float* d_Tc = ctx->d_tmp2.as<float>();
  float* d_Tw = d_Tc + 16 * (size_t)n;
  uint8_t* d_ok = (uint8_t*)(d_Tw + 16 * (size_t)n);
  STOCS_CUDA(ctx, cudaMemcpyAsync(d_b, base_idx4, (size_t)n * 16, cudaMemcpyHostToDevice, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(d_q, quads4, (size_t)n * 16, cudaMemcpyHostToDevice, st));
  FitArgs a;
  fill_fit_args(ctx, a);
  a.base_idx4 = d_b; a.quads4 = d_q; a.Tc = d_Tc; a.Tw = d_Tw; a.ok = d_ok; a.n = n;
  fit_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(a);
  STOCS_CUDA(ctx, cudaGetLastError());
  STOCS_CUDA(ctx, cudaMemcpyAsync(T_centred16, d_Tc, (size_t)n * 64, cudaMemcpyDeviceToHost, st));
  if (T_world16) STOCS_CUDA(ctx, cudaMemcpyAsync(T_world16, d_Tw, (size_t)n * 64, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(ok, d_ok, (size_t)n, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  return STOCS_OK;
}

int stocs_launch_sample_instance(stocs_b200_ctx* ctx, uint64_t seed, int base_num, float dispersion, int* d_ids,
                                 float* d_inv, uint8_t* d_valid, cudaStream_t st);  // sample_instance.cu

// mode 0: class-mode bases (independent, one launch for all); mode 1: instance-mode bases (sequentially
// coupled: one launch per base, base numbers 1..n_bases).  The whole chain -- bases, congruent sets, item
// selection, fits, scores, best, result record -- is enqueued back to back against capacities and the
// host synchronises ONCE, on the 200-byte state record (round 1: six synchronisations per pose).
// cp != NULL: the greedy clustering of the scored list (cluster.cu) is enqueued behind the result record
// and its poses come back in the same queue; with cp == NULL nothing of it is enqueued.
static int run_pipeline_impl(stocs_b200_ctx* ctx, uint64_t seed, int n_bases, int max_sets, int mode, float dispersion,
                             stocs_b200_pipeline_result* result, const stocs_b200_cluster_params* cp = nullptr,
                             stocs_b200_pose* poses = nullptr, int cap = 0, int* n_poses = nullptr) {
  if (!ctx) return STOCS_E_ARG;
  if (cp && (!poses || !n_poses)) STOCS_FAIL(ctx, STOCS_E_ARG, "run_pipeline_clustered: bad argument");
  if (cp && stocs_cluster_check(ctx, cp, cap)) return STOCS_E_ARG;
  if (n_poses) *n_poses = 0;
  if (ctx->S <= 0 || ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "run_pipeline: upload_model and upload_scene first");
  if (n_bases <= 0 || max_sets <= 0 || !result) STOCS_FAIL(ctx, STOCS_E_ARG, "run_pipeline: bad argument");
  if (mode == 1 && n_bases > 255) STOCS_FAIL(ctx, STOCS_E_ARG, "run_pipeline: instance mode numbers its bases 1..255");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  StageTrace tr(st);
  memset(result, 0, sizeof(*result));
  result->best_index = -1;
  result->best_base = -1;
  // 1. bases (rejected ones keep their slot, flagged in d_valid: every later stage skips them, so the
  // order of the valid bases -- base_set of the reference driver -- is preserved without compaction)
  DevBuf& d_bases = ctx->pool[POOL_PIPE_BASES];
  STOCS_CUDA(ctx, d_bases.ensure((size_t)n_bases * 25 + 64));
  int* d_ids = d_bases.as<int>();
  float* d_inv = (float*)(d_ids + 4 * (size_t)n_bases);
  uint8_t* d_valid = (uint8_t*)(d_inv + 2 * (size_t)n_bases);
  int rc = STOCS_OK;
  if (mode == 0) {
    rc = stocs_launch_sample(ctx, seed, 0, n_bases, d_ids, d_inv, d_valid, st);
  } else {
    STOCS_CUDA(ctx, cudaMemsetAsync(d_valid, 0, (size_t)n_bases, st));
    for (int b = 0; b < n_bases && rc == STOCS_OK; ++b)
      rc = stocs_launch_sample_instance(ctx, seed, b + 1, dispersion, d_ids + 4 * (size_t)b, d_inv + 2 * (size_t)b, d_valid + b, st);
  }
  if (rc) return rc;
  tr.mark("pipeline: sample bases");
  DevBuf &d_off = ctx->pool[POOL_PIPE_OFF], &d_items = ctx->pool[POOL_PIPE_ITEMS], &d_fit = ctx->pool[POOL_PIPE_FIT];
  STOCS_CUDA(ctx, ctx->pool[POOL_PIPE_STATE].ensure(sizeof(StocsPipeState)));
  StocsPipeState* d_state = ctx->pool[POOL_PIPE_STATE].as<StocsPipeState>();
  STOCS_CUDA(ctx, d_off.ensure((size_t)(n_bases + 1) * 16));
  long long* d_qoff = d_off.as<long long>();
  long long* d_ioff = d_qoff + (n_bases + 1);
  StocsPipeState& hs = *ctx->h_pipe_state;
  for (int attempt = 0;; ++attempt) {
    STOCS_CUDA(ctx, cudaMemsetAsync(d_state, 0, sizeof(StocsPipeState), st));
    // 2. congruent sets
    rc = stocs_congruent_enqueue(ctx, n_bases, d_ids, d_inv, d_valid, d_state, d_qoff, st);
    if (rc) return rc;
    tr.mark("pipeline: congruent sets");
    // 3. at most max_sets transforms per base; the count is bounded by both n_bases * max_sets and the quad capacity
    long long cap_items = (long long)n_bases * max_sets;
    if (cap_items > ctx->cong_cap_quads) cap_items = ctx->cong_cap_quads;
    pipe_item_offsets_kernel<<<1, 256, 0, st>>>(d_qoff, n_bases, max_sets, d_ioff, d_state);
    STOCS_CUDA(ctx, d_items.ensure((size_t)cap_items * 12));
    long long* d_item_quad = d_items.as<long long>();
    int* d_item_base = (int*)(d_item_quad + cap_items);
    select_items_kernel<<<n_bases, 128, 0, st>>>(d_qoff, d_ioff, n_bases, max_sets, d_item_base, d_item_quad);
    STOCS_CUDA(ctx, d_fit.ensure((size_t)cap_items * (64 + 64 + 1 + 4 + 4) + 1024));
    float* d_Tc = d_fit.as<float>();
    float* d_Tw = d_Tc + 16 * (size_t)cap_items;
    float* d_lcp = d_Tw + 16 * (size_t)cap_items;
    int* d_inl = (int*)(d_lcp + cap_items);
    uint8_t* d_ok = (uint8_t*)(d_inl + cap_items);
    FitArgs a;
    fill_fit_args(ctx, a);
    a.base_idx4 = d_ids; a.quads4 = ctx->pool[POOL_CONG_QUADS].as<int>(); a.item_base = d_item_base; a.item_quad = d_item_quad;
    a.Tc = d_Tc; a.Tw = d_Tw; a.ok = d_ok; a.n = 0; a.n_dev = &d_state->n_items;
    // grids follow the previous run's item count (any grid is correct: the kernels stride / claim up to the device count)
    long long guess = ctx->pipe_last_items > 0 ? ctx->pipe_last_items + ctx->pipe_last_items / 4 : 4096;
    if (guess > cap_items) guess = cap_items;
    if (guess < 1) guess = 1;
    long long fit_blocks = (guess + 127) / 128;
    if (fit_blocks > (long long)ctx->num_sms * 16) fit_blocks = (long long)ctx->num_sms * 16;
    fit_kernel<<<(unsigned)fit_blocks, 128, 0, st>>>(a);
    tr.mark("pipeline: select + fit");
    // 4. score + 5. best
    ScoreRequest sq;
    sq.time_it = true;
    sq.d_H = &d_state->n_items;
    sq.grid_hint = guess;
    rc = stocs_launch_score(ctx, d_Tc, cap_items, d_lcp, d_inl, st, sq);
    if (rc) return rc;
    long long* d_bi = &ctx->scratch()->pipe_best_idx;
    float* d_bv = &ctx->scratch()->pipe_best_lcp;
    // lists the closing block can scan itself (every online frame) skip the general top-K launch
    const bool small_list = cap_items <= (1ll << 20);
    if (!small_list) {
      TopkRequest tq;
      tq.idx = (int64_t*)d_bi;
      tq.val = d_bv;
      tq.d_H = &d_state->n_items;
      tq.grid_hint = guess;
      rc = stocs_launch_topk(ctx, d_lcp, cap_items, 1, 0, st, tq);
      if (rc) return rc;
    }
    pipe_finalize_kernel<<<1, 1024, 0, st>>>(small_list ? d_lcp : nullptr, d_ok, d_valid, n_bases, d_item_base, d_bi, d_bv, d_Tc, d_Tw, d_state);
    STOCS_CUDA(ctx, cudaGetLastError());
    if (cp) {
      const PipeClusterInputs ci = {d_lcp, d_Tc, d_Tw, d_ok, d_valid, d_item_base, cap_items, d_state};
      rc = stocs_cluster_enqueue_pipeline(ctx, *cp, ci, st);
      if (rc) return rc;
    }
    STOCS_CUDA(ctx, cudaMemcpyAsync(&hs, d_state, sizeof(StocsPipeState), cudaMemcpyDeviceToHost, st));
    STOCS_CUDA(ctx, cudaStreamSynchronize(st));
    tr.mark("pipeline: score + best");
    if (!hs.overflow) break;
    if (!stocs_congruent_grow(ctx, hs) || attempt >= 2) STOCS_FAIL(ctx, STOCS_E_ARG, "find_congruent: pair lists too long");
  }
  ctx->pipe_last_items = hs.n_items;
  result->n_valid_bases = hs.n_valid;
  result->n_congruent_sets = (long long)hs.total_quads;
  result->n_transforms = hs.n_ok;
  result->best_lcp = hs.best_lcp;
  if (hs.best_item >= 0) {
    result->best_index = hs.rank_of_best;  // index into the list of pushed transforms, as in the reference
    result->best_base = hs.best_base;
    memcpy(result->best_T_centred, hs.best_Tc, 64);
    memcpy(result->best_T_world, hs.best_Tw, 64);
  }
  if (cp) {
    memcpy(poses, stocs_cluster_poses_host(ctx), (size_t)hs.n_poses * sizeof(stocs_b200_pose));
    *n_poses = hs.n_poses;
  }
  return STOCS_OK;
}

extern "C" int stocs_b200_run_pipeline(stocs_b200_ctx* ctx, uint64_t seed, int n_bases, int max_sets,
                                       stocs_b200_pipeline_result* result) {
  return run_pipeline_impl(ctx, seed, n_bases, max_sets, 0, 0.f, result);
}

extern "C" int stocs_b200_run_pipeline_instance(stocs_b200_ctx* ctx, uint64_t seed, int n_bases, int max_sets,
                                                float dispersion, stocs_b200_pipeline_result* result) {
  return run_pipeline_impl(ctx, seed, n_bases, max_sets, 1, dispersion, result);
}

extern "C" int stocs_b200_run_pipeline_clustered(stocs_b200_ctx* ctx, uint64_t seed, int n_bases, int max_sets,
                                                 const stocs_b200_cluster_params* p, stocs_b200_pipeline_result* result,
                                                 stocs_b200_pose* poses, int cap, int* n_poses) {
  if (!ctx) return STOCS_E_ARG;
  if (!p) STOCS_FAIL(ctx, STOCS_E_ARG, "run_pipeline_clustered: params are NULL");
  return run_pipeline_impl(ctx, seed, n_bases, max_sets, 0, 0.f, result, p, poses, cap, n_poses);
}

extern "C" int stocs_b200_run_pipeline_instance_clustered(stocs_b200_ctx* ctx, uint64_t seed, int n_bases, int max_sets,
                                                          float dispersion, const stocs_b200_cluster_params* p,
                                                          stocs_b200_pipeline_result* result, stocs_b200_pose* poses,
                                                          int cap, int* n_poses) {
  if (!ctx) return STOCS_E_ARG;
  if (!p) STOCS_FAIL(ctx, STOCS_E_ARG, "run_pipeline_clustered: params are NULL");
  return run_pipeline_impl(ctx, seed, n_bases, max_sets, 1, dispersion, result, p, poses, cap, n_poses);
}
