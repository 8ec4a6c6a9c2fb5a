// comm.cu -- hypothesis-sharded scoring across GPUs (SURVEY.md section 8e).
//
// The reference scores every hypothesis in one sequential loop and keeps the first strict maximum
// (src/stocs.cpp:990-998).  Hypotheses are independent, so each GPU scores a contiguous block of
// the list against its own replica of the scene index; the per-GPU K best are packed as 64-byte
// records {lcp, inliers, global index, 3x4 transform} (reduce.cu: topk_kernel), ONE
// ncclAllGather moves nranks*K records (16 KB at 8 GPUs, K = 32) over NVLink, and a single-CTA
// kernel ranks them by (lcp descending, global index ascending): record 0 is the reference's
// winner over the whole list.  The collective is latency-bound; nothing here is worth fusing into
// the scoring kernel (it moves 2 KB per rank once per object).
//
// NCCL is bound at run time (dlopen) so that single-GPU users of libstocs_b200.so do not need it
// and so that a host process that already carries an NCCL (PyTorch bundles its own libnccl.so.2)
// shares that copy instead of loading a second one.
#include <dlfcn.h>
#include <nccl.h>

#include <cstring>
#include <mutex>
#include <new>

#include "stocs_ctx.h"

namespace {

struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string err;
};

NcclApi g_nccl;
std::mutex g_nccl_mu;

// returns NULL on success, else a message
const char* load_nccl() {
  std::lock_guard<std::mutex> lk(g_nccl_mu);
  if (g_nccl.handle) return nullptr;
  const char* names[] = {getenv("STOCS_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) {
    if (!n || !*n) continue;
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) {
    g_nccl.err = std::string("cannot load NCCL (libnccl.so.2; set STOCS_NCCL_LIB): ") + (dlerror() ? dlerror() : "");
    return g_nccl.err.c_str();
  }
  bool ok = true;
  auto sym = [&](const char* s) { void* p = dlsym(h, s); if (!p) { ok = false; g_nccl.err = std::string("NCCL symbol missing: ") + s; } return p; };
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))sym("ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))sym("ncclCommInitRank");
  g_nccl.CommInitAll = (decltype(g_nccl.CommInitAll))sym("ncclCommInitAll");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))sym("ncclCommDestroy");
  g_nccl.AllGather = (decltype(g_nccl.AllGather))sym("ncclAllGather");
  g_nccl.GroupStart = (decltype(g_nccl.GroupStart))sym("ncclGroupStart");
  g_nccl.GroupEnd = (decltype(g_nccl.GroupEnd))sym("ncclGroupEnd");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))sym("ncclGetErrorString");
  if (!ok) { dlclose(h); return g_nccl.err.c_str(); }
  g_nccl.handle = h;
  return nullptr;
}

#define STOCS_NCCL(ctx, call)                                                              \
  do {                                                                                     \
    ncclResult_t _r = (call);                                                              \
    if (_r != ncclSuccess) {                                                               \
      (ctx)->err = std::string(#call) + ": " + g_nccl.GetErrorString(_r);                  \
      return STOCS_E_NCCL;                                                                 \
    }                                                                                      \
  } while (0)

// Rank n records (n <= 2048) by (lcp descending, index ascending), keep the K best.  Every record
// counts the records that beat it; that count is its output slot.  Empty records (index < 0 or
// lcp <= 0) never win; unused output slots are written as empty.  One CTA.
__global__ void __launch_bounds__(1024) merge_records_kernel(const stocs_b200_record* __restrict__ in, int n, int K,
                                                             stocs_b200_record* __restrict__ out) {
  __shared__ float s_lcp[2048];
  __shared__ long long s_idx[2048];
  __shared__ int s_valid;
  if (threadIdx.x == 0) s_valid = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = in[i].lcp;
    const long long ix = in[i].index;
    const bool ok = ix >= 0 && v > 0.f;
    s_lcp[i] = ok ? v : 0.f;
    s_idx[i] = ok ? ix : -1;
    if (ok) atomicAdd(&s_valid, 1);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const long long ix = s_idx[i];
    if (ix < 0) continue;
    const float v = s_lcp[i];
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      const long long jx = s_idx[j];
      if (jx < 0) continue;
      const float w = s_lcp[j];
      rank += (w > v || (w == v && jx < ix)) ? 1 : 0;
    }
    if (rank < K) out[rank] = in[i];
  }
  const int nv = s_valid;
  for (int k = nv + threadIdx.x; k < K; k += blockDim.x) {
    stocs_b200_record r;
    r.lcp = 0.f; r.inliers = 0; r.index = -1;
    for (int t = 0; t < 12; ++t) r.T[t] = 0.f;
    out[k] = r;
  }
}

// local block -> K packed records in d_send (device).  Enqueues on st.
// prune: the caller reads nothing of d_lcp / d_inl but the K records, so hypotheses that provably
// cannot enter the top K may be left unscored (lcp 0, see kPrune in score.cu)
int enqueue_local_topk(stocs_b200_ctx* ctx, const float* d_T, int64_t H_local, int64_t index_offset, int K,
                       float* d_lcp, int32_t* d_inl, stocs_b200_record* d_send, cudaStream_t st, bool time_it, bool prune) {
  ScoreRequest sq;
  sq.time_it = time_it;
  sq.top_K = prune ? K : 0;
  int rc = stocs_launch_score(ctx, d_T, H_local, d_lcp, d_inl, st, sq);
  if (rc) return rc;
  // H_local == 0: nothing is scored, the top-K kernels run over an empty array and emit K empty records
  TopkRequest tq;
  tq.T16 = d_T;
  tq.inl = d_inl;
  tq.rec = d_send;
  return stocs_launch_topk(ctx, d_lcp, H_local, K, index_offset, st, tq);
}

// the buffers of the collective: K local records (POOL_COMM_SEND), nranks*K gathered records
// (POOL_COMM_RECV) and K merged records (POOL_COMM_OUT)
cudaError_t ensure_record_buffers(stocs_b200_ctx* ctx, int K, int nranks) {
  const size_t rec_bytes = (size_t)K * sizeof(stocs_b200_record);
  cudaError_t e = ctx->pool[POOL_COMM_SEND].ensure(rec_bytes);
  if (e == cudaSuccess) e = ctx->pool[POOL_COMM_RECV].ensure(rec_bytes * nranks);
  if (e == cudaSuccess) e = ctx->pool[POOL_COMM_OUT].ensure(rec_bytes);
  return e;
}

// ONE all-gather of the K records every rank left in POOL_COMM_SEND, then their merge into `out`
// (K records), on stream st
int gather_merge_records(stocs_b200_ctx* ctx, int K, stocs_b200_record* out, cudaStream_t st) {
  DevBuf &b_send = ctx->pool[POOL_COMM_SEND], &b_recv = ctx->pool[POOL_COMM_RECV];
  STOCS_NCCL(ctx, g_nccl.AllGather(b_send.p, b_recv.p, (size_t)K * sizeof(stocs_b200_record), ncclInt8,
                                   (ncclComm_t)ctx->comm, st));
  merge_records_kernel<<<1, 1024, 0, st>>>(b_recv.as<stocs_b200_record>(), K * ctx->comm_nranks, K, out);
  STOCS_CUDA(ctx, cudaGetLastError());
  return STOCS_OK;
}

}  // namespace

extern "C" {

void stocs_b200_shard_range(int64_t H, int rank, int nranks, int64_t* lo, int64_t* hi) {
  if (nranks < 1) nranks = 1;
  const int64_t per = (H + nranks - 1) / nranks;
  int64_t a = (int64_t)rank * per;
  if (a > H) a = H;
  int64_t b = a + per;
  if (b > H) b = H;
  if (lo) *lo = a;
  if (hi) *hi = b;
}

int stocs_b200_comm_unique_id(void* id128) {
  if (!id128) return STOCS_E_ARG;
  static_assert(sizeof(ncclUniqueId) == STOCS_B200_UNIQUE_ID_BYTES, "ncclUniqueId is 128 bytes");
  if (load_nccl()) return STOCS_E_NCCL;
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return STOCS_E_NCCL;
  memcpy(id128, &id, sizeof(id));
  return STOCS_OK;
}

int stocs_b200_comm_init(stocs_b200_ctx* ctx, const void* id128, int rank, int nranks) {
  if (!ctx) return STOCS_E_ARG;
  if (!id128 || nranks < 1 || rank < 0 || rank >= nranks) STOCS_FAIL(ctx, STOCS_E_ARG, "comm_init: bad argument");
  if (nranks * 32 > 2048) STOCS_FAIL(ctx, STOCS_E_ARG, "comm_init: at most 64 ranks");
  if (ctx->comm) STOCS_FAIL(ctx, STOCS_E_STATE, "comm_init: communicator already initialised");
  if (const char* e = load_nccl()) STOCS_FAIL(ctx, STOCS_E_NCCL, e);
  cudaSetDevice(ctx->device);
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  ncclComm_t comm = nullptr;
  STOCS_NCCL(ctx, g_nccl.CommInitRank(&comm, nranks, id, rank));
  ctx->comm = comm;
  ctx->comm_rank = rank;
  ctx->comm_nranks = nranks;
  return STOCS_OK;
}

int stocs_b200_comm_destroy(stocs_b200_ctx* ctx) {
  if (!ctx) return STOCS_E_ARG;
  if (ctx->comm) {
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    g_nccl.CommDestroy((ncclComm_t)ctx->comm);
    ctx->comm = nullptr;
  }
  ctx->comm_rank = 0;
  ctx->comm_nranks = 1;
  return STOCS_OK;
}

int stocs_b200_score_sharded_device(stocs_b200_ctx* ctx, const float* d_T16_local, int64_t H_local,
                                    int64_t index_offset, int K, stocs_b200_record* d_topk_out, void* stream) {
  if (!ctx) return STOCS_E_ARG;
  if (ctx->S <= 0 || ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "score_sharded: upload_model and upload_scene first");
  if (H_local < 0 || K < 1 || K > 32 || !d_topk_out || (H_local > 0 && !d_T16_local) || index_offset < 0)
    STOCS_FAIL(ctx, STOCS_E_ARG, "score_sharded: bad argument");
  cudaSetDevice(ctx->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  DevBuf &b_lcp = ctx->pool[POOL_SHARD_LCP], &b_inl = ctx->pool[POOL_SHARD_INL];
  STOCS_CUDA(ctx, b_lcp.ensure((size_t)(H_local ? H_local : 1) * 4));
  STOCS_CUDA(ctx, b_inl.ensure((size_t)(H_local ? H_local : 1) * 4));
  const int nranks = ctx->comm ? ctx->comm_nranks : 1;
  if (nranks == 1)  // no collective: the local top-K is the global one
    return enqueue_local_topk(ctx, d_T16_local, H_local, index_offset, K, b_lcp.as<float>(), b_inl.as<int32_t>(),
                              d_topk_out, st, true, true);
  STOCS_CUDA(ctx, ensure_record_buffers(ctx, K, nranks));
  int rc = enqueue_local_topk(ctx, d_T16_local, H_local, index_offset, K, b_lcp.as<float>(), b_inl.as<int32_t>(),
                              ctx->pool[POOL_COMM_SEND].as<stocs_b200_record>(), st, true, true);
  if (rc) return rc;
  return gather_merge_records(ctx, K, d_topk_out, st);
}

int stocs_b200_score_sharded(stocs_b200_ctx* ctx, const float* T16_local, int64_t H_local, int64_t index_offset, int K,
                             stocs_b200_record* topk_out, float* lcp_local, int32_t* inliers_local) {
  if (!ctx) return STOCS_E_ARG;
  if (H_local < 0 || K < 1 || K > 32 || !topk_out || (H_local > 0 && !T16_local) || index_offset < 0)
    STOCS_FAIL(ctx, STOCS_E_ARG, "score_sharded: bad argument");
  if (ctx->S <= 0 || ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "score_sharded: upload_model and upload_scene first");
  cudaSetDevice(ctx->device);
  const int nranks = ctx->comm ? ctx->comm_nranks : 1;
  STOCS_CUDA(ctx, ensure_record_buffers(ctx, K, nranks));
  stocs_b200_record* d_out = ctx->pool[POOL_COMM_OUT].as<stocs_b200_record>();
  stocs_b200_record* d_local = nranks > 1 ? ctx->pool[POOL_COMM_SEND].as<stocs_b200_record>() : d_out;
  // ONE pass with ONE synchronisation: the records are the tail of the host-buffer scoring call --
  // the K best of the resident results as records, ONE all-gather and the merge, the K merged
  // records back.  (Scoring through the single-GPU host call first, with its own top-32 reduction
  // and synchronisation, cost 0.58 against 0.50 ms per step at 125 000 hypotheses per rank on 8 GPUs.)
  auto tail = [&](cudaStream_t st, const float* d_T) -> int {
    TopkRequest tq;
    tq.T16 = d_T;
    tq.inl = ctx->d_inl.as<int32_t>();
    tq.rec = d_local;
    int rc = stocs_launch_topk(ctx, ctx->d_lcp.as<float>(), H_local, K, index_offset, st, tq);
    if (rc == STOCS_OK && nranks > 1) rc = gather_merge_records(ctx, K, d_out, st);
    if (rc) return rc;
    STOCS_CUDA(ctx, cudaMemcpyAsync(topk_out, d_out, (size_t)K * sizeof(stocs_b200_record), cudaMemcpyDeviceToHost, st));
    return STOCS_OK;
  };
  return stocs_score_host(ctx, "score_sharded", T16_local, H_local, lcp_local, inliers_local, tail);
}

}  // extern "C"

// ---- single-process group -----------------------------------------------------------------------
struct stocs_b200_group {
  std::vector<stocs_b200_ctx*> ctx;
  std::string err;
};

static int group_fail(stocs_b200_group* g, int i, int rc) {
  g->err = "device " + std::to_string(g->ctx[i]->device) + ": " + stocs_b200_last_error(g->ctx[i]);
  return rc;
}

extern "C" {

int stocs_b200_group_create(stocs_b200_group** out, const int* device_ids, int n_dev) {
  if (!out || !device_ids || n_dev < 1 || n_dev > 64) return STOCS_E_ARG;
  *out = nullptr;
  stocs_b200_group* g = new (std::nothrow) stocs_b200_group();
  if (!g) return STOCS_E_ARG;
  for (int i = 0; i < n_dev; ++i) {
    stocs_b200_ctx* c = nullptr;
    int rc = stocs_b200_create(&c, device_ids[i]);
    if (rc != STOCS_OK) { stocs_b200_group_destroy(g); return rc; }
    g->ctx.push_back(c);
  }
  if (n_dev > 1) {
    if (load_nccl()) { stocs_b200_group_destroy(g); return STOCS_E_NCCL; }
    std::vector<ncclComm_t> comms((size_t)n_dev);
    if (g_nccl.CommInitAll(comms.data(), n_dev, device_ids) != ncclSuccess) { stocs_b200_group_destroy(g); return STOCS_E_NCCL; }
    for (int i = 0; i < n_dev; ++i) {
      g->ctx[i]->comm = comms[i];
      g->ctx[i]->comm_rank = i;
      g->ctx[i]->comm_nranks = n_dev;
    }
  }
  *out = g;
  return STOCS_OK;
}

void stocs_b200_group_destroy(stocs_b200_group* g) {
  if (!g) return;
  for (stocs_b200_ctx* c : g->ctx) { stocs_b200_comm_destroy(c); stocs_b200_destroy(c); }
  delete g;
}

int stocs_b200_group_size(stocs_b200_group* g) { return g ? (int)g->ctx.size() : 0; }
stocs_b200_ctx* stocs_b200_group_ctx(stocs_b200_group* g, int i) {
  return (g && i >= 0 && i < (int)g->ctx.size()) ? g->ctx[i] : nullptr;
}
const char* stocs_b200_group_last_error(stocs_b200_group* g) { return g ? g->err.c_str() : "no group"; }

int stocs_b200_group_set_params(stocs_b200_group* g, float distance_threshold, int tr, int rot) {
  if (!g) return STOCS_E_ARG;
  for (size_t i = 0; i < g->ctx.size(); ++i) {
    int rc = stocs_b200_set_params(g->ctx[i], distance_threshold, tr, rot);
    if (rc) return group_fail(g, (int)i, rc);
  }
  return STOCS_OK;
}

int stocs_b200_group_upload_model(stocs_b200_group* g, const float* pos3, const float* nrm3, int M) {
  if (!g) return STOCS_E_ARG;
  for (size_t i = 0; i < g->ctx.size(); ++i) {
    int rc = stocs_b200_upload_model(g->ctx[i], pos3, nrm3, M);
    if (rc) return group_fail(g, (int)i, rc);
  }
  return STOCS_OK;
}

int stocs_b200_group_upload_scene(stocs_b200_group* g, const float* pos3, const float* nrm3, const float* cls,
                                  const int32_t* pixel_rc, int S) {
  if (!g) return STOCS_E_ARG;
  for (size_t i = 0; i < g->ctx.size(); ++i) {
    int rc = stocs_b200_upload_scene(g->ctx[i], pos3, nrm3, cls, pixel_rc, S);
    if (rc) return group_fail(g, (int)i, rc);
  }
  return STOCS_OK;
}

int stocs_b200_group_score_best(stocs_b200_group* g, const float* T16, int64_t H, int K, stocs_b200_record* topk_out,
                                float* lcp, int32_t* inliers) {
  if (!g || g->ctx.empty()) return STOCS_E_ARG;
  if (H < 0 || K < 1 || K > 32 || !topk_out || (H > 0 && !T16)) { g->err = "group_score_best: bad argument"; return STOCS_E_ARG; }
  const int n = (int)g->ctx.size();
  const size_t rec_bytes = (size_t)K * sizeof(stocs_b200_record);
  std::vector<int64_t> lo((size_t)n), hi((size_t)n);
  // 1. every device: stage its block, score, local top-K records (all asynchronous)
  for (int i = 0; i < n; ++i) {
    stocs_b200_ctx* c = g->ctx[i];
    if (c->S <= 0 || c->M <= 0) { g->err = "group_score_best: upload_model and upload_scene first"; return STOCS_E_STATE; }
    stocs_b200_shard_range(H, i, n, &lo[i], &hi[i]);
    const int64_t hl = hi[i] - lo[i];
    cudaSetDevice(c->device);
    cudaStream_t st = c->stream;
    DevBuf &b_T = c->pool[POOL_SHARD_T], &b_lcp = c->pool[POOL_SHARD_LCP], &b_inl = c->pool[POOL_SHARD_INL];
    cudaError_t e = b_T.ensure((size_t)(hl ? hl : 1) * 64);
    if (e == cudaSuccess) e = b_lcp.ensure((size_t)(hl ? hl : 1) * 4);
    if (e == cudaSuccess) e = b_inl.ensure((size_t)(hl ? hl : 1) * 4);
    if (e == cudaSuccess) e = ensure_record_buffers(c, K, n);
    if (e == cudaSuccess && hl > 0)
      e = cudaMemcpyAsync(b_T.p, T16 + 16 * lo[i], (size_t)hl * 64, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) { c->err = std::string("group_score_best: ") + cudaGetErrorString(e); return group_fail(g, i, STOCS_E_CUDA); }
    int rc = enqueue_local_topk(c, b_T.as<float>(), hl, lo[i], K, b_lcp.as<float>(), b_inl.as<int32_t>(),
                                c->pool[n > 1 ? POOL_COMM_SEND : POOL_COMM_OUT].as<stocs_b200_record>(), st, false,
                                !lcp && !inliers);
    if (rc) return group_fail(g, i, rc);
  }
  // 2. ONE all-gather (grouped: one call per device of this process)
  if (n > 1) {
    if (g_nccl.GroupStart() != ncclSuccess) { g->err = "ncclGroupStart failed"; return STOCS_E_NCCL; }
    for (int i = 0; i < n; ++i) {
      stocs_b200_ctx* c = g->ctx[i];
      ncclResult_t r = g_nccl.AllGather(c->pool[POOL_COMM_SEND].p, c->pool[POOL_COMM_RECV].p, rec_bytes, ncclInt8,
                                        (ncclComm_t)c->comm, c->stream);
      if (r != ncclSuccess) { g_nccl.GroupEnd(); g->err = std::string("ncclAllGather: ") + g_nccl.GetErrorString(r); return STOCS_E_NCCL; }
    }
    if (g_nccl.GroupEnd() != ncclSuccess) { g->err = "ncclGroupEnd failed"; return STOCS_E_NCCL; }
    // 3. merge (device 0 is the one whose answer is returned; every device holds the same records)
    stocs_b200_ctx* c0 = g->ctx[0];
    cudaSetDevice(c0->device);
    merge_records_kernel<<<1, 1024, 0, c0->stream>>>(c0->pool[POOL_COMM_RECV].as<stocs_b200_record>(), K * n, K,
                                                     c0->pool[POOL_COMM_OUT].as<stocs_b200_record>());
  }
  // 4. results
  for (int i = 0; i < n; ++i) {
    stocs_b200_ctx* c = g->ctx[i];
    const int64_t hl = hi[i] - lo[i];
    cudaSetDevice(c->device);
    cudaError_t e = cudaSuccess;
    if (i == 0) e = cudaMemcpyAsync(topk_out, c->pool[POOL_COMM_OUT].p, rec_bytes, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess && lcp && hl > 0)
      e = cudaMemcpyAsync(lcp + lo[i], c->pool[POOL_SHARD_LCP].p, (size_t)hl * 4, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess && inliers && hl > 0)
      e = cudaMemcpyAsync(inliers + lo[i], c->pool[POOL_SHARD_INL].p, (size_t)hl * 4, cudaMemcpyDeviceToHost, c->stream);
    if (e != cudaSuccess) { c->err = std::string("group_score_best: ") + cudaGetErrorString(e); return group_fail(g, i, STOCS_E_CUDA); }
  }
  for (int i = 0; i < n; ++i) {
    stocs_b200_ctx* c = g->ctx[i];
    cudaSetDevice(c->device);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { c->err = std::string("group_score_best: ") + cudaGetErrorString(e); return group_fail(g, i, STOCS_E_CUDA); }
  }
  return STOCS_OK;
}

}  // extern "C"
