// capi.cu -- the C ABI of libstocs_b200.so (include/stocs_b200.h): context, uploads, host-buffer
// wrappers around the kernels.  No CPU fallback anywhere: every compute entry point launches
// sm_100a kernels, and stocs_b200_create refuses to run without a compute-capability-10 device.
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "stocs_ctx.h"

int stocs_build_ppf_table(stocs_b200_ctx* ctx);                         // ppf_table.cu

// "acos(d)*180/pi < 30" (src/stocs.cpp:1028-1032) is monotone in d: find the smallest binary32 d
// for which it holds by bisection over bit patterns, using the same math header as the oracle.
float stocs_angle_threshold_dot() {
  auto pred = [](float d) { return (float)stocsm::rad_to_deg_ref(stocsm::acos_f(d)) < 30.0f; };
  uint32_t lo = stocsm::fbits(0.0f), hi = stocsm::fbits(1.0f);
  while (hi - lo > 1) {
    uint32_t mid = lo + (hi - lo) / 2;
    if (pred(stocsm::bitsf(mid))) hi = mid; else lo = mid;
  }
  return stocsm::bitsf(hi);
}

static thread_local std::string g_create_err;

// Page-locked host memory (cudaHostAlloc / cudaHostRegister, e.g. a pinned torch tensor) is mapped
// into the device address space; this is its device alias, NULL for any other pointer.
const void* stocs_host_alias(const void* p) {
  cudaPointerAttributes pa{};
  if (cudaPointerGetAttributes(&pa, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return pa.type == cudaMemoryTypeHost ? pa.devicePointer : nullptr;
}

// The host-buffer scoring calls read page-locked transforms in place through their device alias;
// NULL: stage them through HBM (pageable memory, or STOCS_NO_ZERO_COPY set).
const float* stocs_zero_copy_transforms(const float* T16) {
  if (getenv("STOCS_NO_ZERO_COPY")) return nullptr;
  return (const float*)stocs_host_alias(T16);
}

// Largest class weight of the scene.  The top-K pruning bound of the scoring kernel (score.cu) needs
// every weight of the scene in [0, w_max]; whatever replaces the weights calls this again.
void stocs_set_weight_bound(stocs_b200_ctx* ctx, const float* cls, int S) {
  ctx->w_max = 0.f;
  ctx->prune_ok = true;
  for (int i = 0; i < S; ++i) {
    const float w = cls[i];
    if (!(w >= 0.f && w <= FLT_MAX)) { ctx->prune_ok = false; break; }   // negative, NaN or infinite
    if (w > ctx->w_max) ctx->w_max = w;
  }
}

// Top-32 of the resident lcp array into the page-locked cache, on stream st (no synchronize).
static int enqueue_resident_topk(stocs_b200_ctx* ctx, int64_t H, cudaStream_t st) {
  DevBuf& d_top = ctx->pool[POOL_TOPK_RESIDENT];
  STOCS_CUDA(ctx, d_top.ensure(32 * 12));
  TopkRequest rq;
  rq.idx = d_top.as<int64_t>();
  rq.val = (float*)(rq.idx + 32);
  int rc = stocs_launch_topk(ctx, ctx->d_lcp.as<float>(), H, 32, 0, st, rq);
  if (rc) return rc;
  STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->h_top->idx, rq.idx, 32 * 8, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->h_top->val, rq.val, 32 * 4, cudaMemcpyDeviceToHost, st));
  return STOCS_OK;
}

int stocs_score_host(stocs_b200_ctx* ctx, const char* who, const float* T16, int64_t H, float* lcp, int32_t* inliers,
                     const ScoreTail& tail) {
  cudaStream_t st = ctx->stream, aux = ctx->aux_stream;
  int rc = STOCS_OK;
  cudaError_t e = cudaSuccess;
  auto ok = [&]() { return rc == STOCS_OK && e == cudaSuccess; };
  // The second stream starts behind whatever is queued on the context stream; once forked, it is
  // joined back even after an error, so that no work is left queued behind the context stream
  // (the one callers order against).
  bool forked = false;
  auto fork = [&]() {
    forked = true;
    e = cudaEventRecord(ctx->join_ev[0], st);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(aux, ctx->join_ev[0], 0);
  };
  auto join = [&]() {
    cudaError_t e2 = cudaEventRecord(ctx->join_ev[1], aux);
    if (e2 == cudaSuccess) e2 = cudaStreamWaitEvent(st, ctx->join_ev[1], 0);
    if (e == cudaSuccess) e = e2;
  };
  if (H == 0) {
    rc = tail(st, nullptr);
  } else {
    ctx->top_valid = false;
    e = ctx->d_lcp.ensure((size_t)H * 4);
    if (e == cudaSuccess) e = ctx->d_inl.ensure((size_t)H * 4);
    float* d_lcp = ctx->d_lcp.as<float>();
    int32_t* d_inl = ctx->d_inl.as<int32_t>();
    // Page-locked, device-mapped transforms (cudaHostAlloc / cudaHostRegister, e.g. a pinned torch
    // tensor) are read by the kernel in place: each warp fetches its 48 B over PCIe while the SM's
    // other 63 warps compute, so no staging copy and a single launch (one straggler tail instead of
    // one per chunk).  Measured on S1: 2.98 ms against 2.94 ms with the transforms in HBM; when every
    // hypothesis is trivially rejected the reads become the bound (1.56 ms per 10^6, 41 GB/s), still
    // no slower than the staged path.  Results are written to HBM and copied back once: letting the
    // kernel also write to host memory puts its reads behind the posted writes (3.98 ms).
    if (const float* d_T = ok() ? stocs_zero_copy_transforms(T16) : nullptr) {
      ScoreRequest rq;
      rq.time_it = true;
      rc = stocs_launch_score(ctx, d_T, H, d_lcp, d_inl, st, rq);
      // the tail runs on the second stream while the copy engine returns the results
      if (ok()) fork();
      if (ok() && lcp) e = cudaMemcpyAsync(lcp, d_lcp, (size_t)H * 4, cudaMemcpyDeviceToHost, st);
      if (ok() && inliers) e = cudaMemcpyAsync(inliers, d_inl, (size_t)H * 4, cudaMemcpyDeviceToHost, st);
      if (ok()) rc = tail(aux, d_T);
      if (forked) join();
    } else {
      // Pageable transforms are staged through HBM in chunks: the H2D copy of chunk k+1 (copy
      // stream) overlaps the scoring of chunk k.  Chunks grow geometrically (H/8, H/8, H/4, H/2) so
      // that scoring starts early and most of the work runs in large launches.  Consecutive chunks
      // alternate between two compute streams, each launch with its own work counter, so the CTAs
      // of chunk k+1 move in as the straggler warps of chunk k retire (a launch's tail is 0.1-0.2 ms
      // on the S1 workload); each chunk's results go back on its own stream behind its kernel.
      // (H2D from pageable memory is staged by the driver through its own pinned buffer and returns
      // early; D2H into pageable memory does not -- see below.)
      if (ok()) e = ctx->d_T.ensure((size_t)H * 64);
      float* d_stage = ctx->d_T.as<float>();
      std::vector<int64_t> bounds;
      if (H <= (1 << 16)) {
        bounds = {0, H};
      } else {
        const int64_t e8 = (H + 7) / 8;
        bounds = {0, e8, 2 * e8, 4 * e8, H};
        for (auto& b : bounds) if (b > H) b = H;
      }
      const int64_t nchunks = (int64_t)bounds.size() - 1;
      cudaStream_t cs[2] = {st, aux};
      if (ok() && nchunks > 1) fork();
      for (int64_t c = 0; c < nchunks && ok(); ++c) {
        const int64_t off = bounds[c], n = bounds[c + 1] - bounds[c];
        if (n <= 0) continue;
        e = cudaMemcpyAsync(d_stage + off * 16, T16 + off * 16, (size_t)n * 64, cudaMemcpyHostToDevice, ctx->copy_stream);
        if (e == cudaSuccess) e = cudaEventRecord(ctx->chunk_ev[c], ctx->copy_stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(cs[c & 1], ctx->chunk_ev[c], 0);
        ScoreRequest rq;
        rq.slot = (int)c;
        if (e == cudaSuccess) rc = stocs_launch_score(ctx, d_stage + off * 16, n, d_lcp + off, d_inl + off, cs[c & 1], rq);
      }
      // Result copies are enqueued only after EVERY chunk's H2D copy and kernel: a cudaMemcpyAsync
      // into pageable memory returns when the copy is done, so issuing it inside the loop above would
      // hold back the enqueue of chunk k+1's H2D until chunk k's kernel has finished (no overlap at all).
      for (int64_t c = 0; c < nchunks && ok(); ++c) {
        const int64_t off = bounds[c], n = bounds[c + 1] - bounds[c];
        if (n <= 0) continue;
        if (lcp) e = cudaMemcpyAsync(lcp + off, d_lcp + off, (size_t)n * 4, cudaMemcpyDeviceToHost, cs[c & 1]);
        if (e == cudaSuccess && inliers)
          e = cudaMemcpyAsync(inliers + off, d_inl + off, (size_t)n * 4, cudaMemcpyDeviceToHost, cs[c & 1]);
      }
      if (forked) join();
      if (ok()) rc = tail(st, d_stage);
    }
  }
  const cudaError_t es = cudaStreamSynchronize(st);
  if (e == cudaSuccess) e = es;
  if (rc == STOCS_OK && e != cudaSuccess) { ctx->err = std::string(who) + ": " + cudaGetErrorString(e); rc = STOCS_E_CUDA; }
  if (H > 0) ctx->last_H = rc == STOCS_OK ? H : 0;
  return rc;
}

extern "C" {

int stocs_b200_abi_version(void) { return STOCS_B200_ABI_VERSION; }

int stocs_b200_create(stocs_b200_ctx** out, int device) {
  if (!out) return STOCS_E_ARG;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) {
    g_create_err = std::string("no CUDA device: ") + cudaGetErrorString(e);
    return STOCS_E_NODEVICE;
  }
  if (device < 0 || device >= ndev) { g_create_err = "bad device ordinal"; return STOCS_E_ARG; }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return STOCS_E_CUDA;
  if (prop.major != 10) {
    g_create_err = "libstocs_b200 is built for sm_100a only; device is sm_" + std::to_string(prop.major) +
                   std::to_string(prop.minor);
    return STOCS_E_NODEVICE;
  }
  if (cudaSetDevice(device) != cudaSuccess) return STOCS_E_CUDA;
  stocs_b200_ctx* ctx = new (std::nothrow) stocs_b200_ctx();
  if (!ctx) return STOCS_E_ARG;
  ctx->device = device;
  ctx->num_sms = prop.multiProcessorCount;
  bool ok = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&ctx->join_ev[0], cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&ctx->join_ev[1], cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaHostAlloc((void**)&ctx->h_top, sizeof(stocs_b200_ctx::TopCache), cudaHostAllocDefault) == cudaSuccess;
  ok = ok && cudaHostAlloc((void**)&ctx->h_pipe_state, sizeof(StocsPipeState), cudaHostAllocDefault) == cudaSuccess;
  ok = ok && cudaHostAlloc((void**)&ctx->h_index_counts, 4 * (8 + 1 + STOCS_B200_MAX_CLOUD_OBJECTS), cudaHostAllocDefault) == cudaSuccess;
  for (int i = 0; ok && i < stocs_b200_ctx::kMaxChunks; ++i)
    ok = cudaEventCreateWithFlags(&ctx->chunk_ev[i], cudaEventDisableTiming) == cudaSuccess;
  if (!ok) { g_create_err = "stream/event creation failed"; delete ctx; return STOCS_E_CUDA; }
  ctx->dot_thr = stocs_angle_threshold_dot();
  // initial capacities of the online stages (tests shrink them to exercise the grow-and-retry path)
  if (const char* e = getenv("STOCS_CONG_CAP_CODES")) { const long long v = atoll(e); if (v >= 1 && v < (1ll << 31)) ctx->cong_cap_codes = v; }
  if (const char* e = getenv("STOCS_CONG_CAP_QUADS")) { const long long v = atoll(e); if (v >= 1 && v < (1ll << 31)) ctx->cong_cap_quads = v; }
  if (ctx->d_small.ensure(4096) != cudaSuccess || cudaMemset(ctx->d_small.p, 0, 4096) != cudaSuccess) {
    g_create_err = "device allocation failed";
    stocs_b200_destroy(ctx);
    return STOCS_E_CUDA;
  }
  if (!stocs_fmad_selftest(ctx)) {
    g_create_err = "self-test failed: kernels were built with fused multiply-add contraction";
    stocs_b200_destroy(ctx);
    return STOCS_E_CUDA;
  }
  *out = ctx;
  return STOCS_OK;
}

void stocs_b200_destroy(stocs_b200_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  stocs_kd_finish(ctx, ctx->stream, false);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  stocs_b200_comm_destroy(ctx);
  DevBuf* bufs[] = {&ctx->d_model, &ctx->d_mpos4, &ctx->d_mnrm4, &ctx->d_spos4, &ctx->d_sattr, &ctx->d_spix,
                    &ctx->d_coarse, &ctx->d_brick_occ, &ctx->d_bricks, &ctx->d_cell_start, &ctx->d_cand, &ctx->d_kd_nodes, &ctx->d_kd_pts, &ctx->d_ppf_bin_start,
                    &ctx->d_ppf_pairs, &ctx->d_ppf_keybits, &ctx->d_T, &ctx->d_lcp, &ctx->d_inl, &ctx->d_work,
                    &ctx->d_tmp, &ctx->d_tmp2, &ctx->d_small, &ctx->d_edge, &ctx->d_inst_state, &ctx->d_mask_store,
                    &ctx->d_frontier};
  for (DevBuf* b : bufs) b->release();
  for (DevBuf& b : ctx->pool) b.release();
  for (cudaEvent_t e : ctx->ev_ring) if (e) cudaEventDestroy(e);
  for (int i = 0; i < stocs_b200_ctx::kMaxChunks; ++i) if (ctx->chunk_ev[i]) cudaEventDestroy(ctx->chunk_ev[i]);
  for (int i = 0; i < 2; ++i) if (ctx->join_ev[i]) cudaEventDestroy(ctx->join_ev[i]);
  if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
  if (ctx->h_top) cudaFreeHost(ctx->h_top);
  if (ctx->h_pipe_state) cudaFreeHost(ctx->h_pipe_state);
  stocs_cluster_free_host(ctx);
  if (ctx->h_index_counts) cudaFreeHost(ctx->h_index_counts);
  if (ctx->h_kd_stage) cudaFreeHost(ctx->h_kd_stage);
  if (ctx->kd_copy_done) cudaEventDestroy(ctx->kd_copy_done);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  delete ctx;
}

const char* stocs_b200_last_error(stocs_b200_ctx* ctx) {
  if (!ctx) return g_create_err.c_str();
  return ctx->err.c_str();
}

int stocs_b200_set_params(stocs_b200_ctx* ctx, float distance_threshold, int tr, int rot) {
  if (!ctx) return STOCS_E_ARG;
  if (!(distance_threshold > 0.f) || tr <= 0 || rot <= 0) STOCS_FAIL(ctx, STOCS_E_ARG, "set_params: bad value");
  if (ctx->S > 0 || ctx->M > 0) STOCS_FAIL(ctx, STOCS_E_STATE, "set_params must precede upload_model/upload_scene");
  ctx->eps = distance_threshold;
  ctx->tr = tr;
  ctx->rot = rot;
  return STOCS_OK;
}

int stocs_b200_backproject(stocs_b200_ctx* ctx, const uint16_t* depth, const uint8_t* bgr, int W, int H,
                           float fx, float cx, float fy, float cy, float depth_scale, float* xyz_out,
                           uint32_t* rgb_out) {
  if (!ctx) return STOCS_E_ARG;
  if (!depth || !xyz_out || W <= 0 || H <= 0) STOCS_FAIL(ctx, STOCS_E_ARG, "backproject: bad argument");
  cudaSetDevice(ctx->device);
  const size_t n = (size_t)W * H;
  const bool color = bgr && rgb_out;
  // layout in d_tmp: depth (2n) | bgr (3n) ; d_tmp2: xyz (12n) | rgb (4n)
  STOCS_CUDA(ctx, ctx->d_tmp.ensure(n * 2 + n * 3 + 64));
  STOCS_CUDA(ctx, ctx->d_tmp2.ensure(n * 12 + n * 4));
  uint16_t* d_depth = ctx->d_tmp.as<uint16_t>();
  uint8_t* d_bgr = ctx->d_tmp.as<uint8_t>() + ((n * 2 + 15) / 16) * 16;
  float* d_xyz = ctx->d_tmp2.as<float>();
  uint32_t* d_rgb = (uint32_t*)(ctx->d_tmp2.as<char>() + n * 12);
  cudaStream_t st = ctx->stream;
  STOCS_CUDA(ctx, cudaMemcpyAsync(d_depth, depth, n * 2, cudaMemcpyHostToDevice, st));
  if (color) STOCS_CUDA(ctx, cudaMemcpyAsync(d_bgr, bgr, n * 3, cudaMemcpyHostToDevice, st));
  int rc = stocs_launch_backproject(ctx, d_depth, color ? d_bgr : nullptr, W, H, fx, cx, fy, cy, depth_scale,
                                    d_xyz, color ? d_rgb : nullptr, st);
  if (rc) return rc;
  STOCS_CUDA(ctx, cudaMemcpyAsync(xyz_out, d_xyz, n * 12, cudaMemcpyDeviceToHost, st));
  if (color) STOCS_CUDA(ctx, cudaMemcpyAsync(rgb_out, d_rgb, n * 4, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  return STOCS_OK;
}

int stocs_b200_upload_model(stocs_b200_ctx* ctx, const float* pos3, const float* nrm3, int M) {
  if (!ctx) return STOCS_E_ARG;
  if (!pos3 || !nrm3 || M <= 0) STOCS_FAIL(ctx, STOCS_E_ARG, "upload_model: bad argument");
  if (M > 5120) STOCS_FAIL(ctx, STOCS_E_ARG, "upload_model: at most 5120 model points are supported");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  STOCS_CUDA(ctx, ctx->d_tmp.ensure((size_t)M * 12));
  STOCS_CUDA(ctx, ctx->d_tmp2.ensure((size_t)M * 12));
  STOCS_CUDA(ctx, ctx->d_mpos4.ensure((size_t)M * 16));
  STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->d_tmp.p, pos3, (size_t)M * 12, cudaMemcpyHostToDevice, st));
  // centroid, centred copy and box on the host (see stocs_centre_points); the device centres its own copy
  ctx->h_mpos.resize((size_t)M * 3);
  int rc = stocs_centre_points(ctx, ctx->d_tmp.as<float>(), M, ctx->d_mpos4.as<float4>(), nullptr, ctx->cm, nullptr, pos3,
                               ctx->h_mpos.data());
  if (rc) return rc;
  ctx->h_mnrm.assign(nrm3, nrm3 + (size_t)M * 3);
  const int Mpad = ((M + 63) / 64) * 64;  // the scoring kernel consumes 64 points per iteration
  // scoring-kernel layout: float4 centred positions (4*Mpad floats), then float4 normals
  std::vector<float> soa((size_t)8 * Mpad, 0.f);
  for (int i = M; i < Mpad; ++i)   // padding points are NaN: they fall outside every grid
    for (int k = 0; k < 3; ++k) soa[4 * (size_t)i + k] = std::nanf("");
  std::vector<float> n4((size_t)4 * M, 0.f);
  for (int i = 0; i < M; ++i)
    for (int k = 0; k < 3; ++k) {
      soa[4 * (size_t)i + k] = ctx->h_mpos[3 * (size_t)i + k];
      soa[4 * (size_t)(Mpad + i) + k] = nrm3[3 * (size_t)i + k];
      n4[4 * (size_t)i + k] = nrm3[3 * (size_t)i + k];
    }
  STOCS_CUDA(ctx, ctx->d_model.ensure(soa.size() * 4));
  STOCS_CUDA(ctx, ctx->d_mnrm4.ensure(n4.size() * 4));
  STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->d_model.p, soa.data(), soa.size() * 4, cudaMemcpyHostToDevice, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->d_mnrm4.p, n4.data(), n4.size() * 4, cudaMemcpyHostToDevice, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->M = M;
  ctx->Mpad = Mpad;
  return stocs_build_ppf_table(ctx);
}

int stocs_b200_upload_scene(stocs_b200_ctx* ctx, const float* pos3, const float* nrm3,
                            const float* class_probability, const int32_t* pixel_rc, int S) {
  if (!ctx) return STOCS_E_ARG;
  if (!pos3 || !nrm3 || !class_probability || S <= 0) STOCS_FAIL(ctx, STOCS_E_ARG, "upload_scene: bad argument");
  if (S > (1 << 27)) STOCS_FAIL(ctx, STOCS_E_ARG, "upload_scene: at most 2^27 scene points are supported");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  // The previous scene is invalid from here on; S is committed only when the new index is complete,
  // so an early error return cannot leave S > 0 describing buffers that were half replaced.
  ctx->S = 0;
  ctx->S_pending = S;
  stocs_kd_finish(ctx, st, false);   // a kd-tree still being built belongs to the scene this call replaces
  // attributes: d_tmp = nrm3 | cls
  STOCS_CUDA(ctx, ctx->d_tmp.ensure((size_t)S * 16));
  float* d_n = ctx->d_tmp.as<float>();
  float* d_c = d_n + (size_t)S * 3;
  STOCS_CUDA(ctx, cudaMemcpyAsync(d_n, nrm3, (size_t)S * 12, cudaMemcpyHostToDevice, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(d_c, class_probability, (size_t)S * 4, cudaMemcpyHostToDevice, st));
  int rc = stocs_pack_scene_attr(ctx, d_n, d_c, S);
  if (rc) { ctx->S_pending = 0; return rc; }
  // (no synchronisation: the position upload below re-uses d_tmp in stream order, and the H2D copies
  // of pageable host memory have consumed their source buffers when cudaMemcpyAsync returns)
  STOCS_CUDA(ctx, ctx->d_spix.ensure((size_t)S * 8));
  if (pixel_rc) STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->d_spix.p, pixel_rc, (size_t)S * 8, cudaMemcpyHostToDevice, st));
  else STOCS_CUDA(ctx, cudaMemsetAsync(ctx->d_spix.p, 0, (size_t)S * 8, st));
  ctx->has_pixels = pixel_rc != nullptr;
  stocs_set_weight_bound(ctx, class_probability, S);
  ctx->pix_min[0] = ctx->pix_min[1] = 0; ctx->pix_max[0] = ctx->pix_max[1] = 0;
  if (pixel_rc) {  // range of the pixel coordinates: instance sampling indexes images with them
    ctx->pix_min[0] = ctx->pix_max[0] = pixel_rc[0]; ctx->pix_min[1] = ctx->pix_max[1] = pixel_rc[1];
    for (int i = 0; i < S; ++i)
      for (int k = 0; k < 2; ++k) {
        const int v = pixel_rc[2 * (size_t)i + k];
        if (v < ctx->pix_min[k]) ctx->pix_min[k] = v;
        if (v > ctx->pix_max[k]) ctx->pix_max[k] = v;
      }
  }
  if (ctx->d_inst_state.p)  // a new scene starts with empty previous_segment / segmentation_buffer
    STOCS_CUDA(ctx, cudaMemsetAsync(ctx->d_inst_state.p, 0, (size_t)ctx->img_w * ctx->img_h * 3, st));
  // positions -> centre -> index
  STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->d_tmp.p, pos3, (size_t)S * 12, cudaMemcpyHostToDevice, st));
  ctx->h_pos_pending = getenv("STOCS_DEVICE_CENTROID") ? nullptr : pos3;
  rc = stocs_build_scene_index(ctx);
  ctx->h_pos_pending = nullptr;
  ctx->S_pending = 0;
  if (rc) { ctx->S = 0; return rc; }
  ctx->S = S;
  return STOCS_OK;
}

int stocs_b200_get_centroids(stocs_b200_ctx* ctx, float* scene3, float* model3) {
  if (!ctx) return STOCS_E_ARG;
  if (scene3) { if (ctx->S <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "no scene"); memcpy(scene3, ctx->cs, 12); }
  if (model3) { if (ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "no model"); memcpy(model3, ctx->cm, 12); }
  return STOCS_OK;
}

int stocs_b200_get_centred(stocs_b200_ctx* ctx, float* scene_pos3, float* model_pos3) {
  if (!ctx) return STOCS_E_ARG;
  if (scene_pos3) {
    if (ctx->S <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "no scene");
    memcpy(scene_pos3, ctx->h_spos.data(), (size_t)ctx->S * 12);
  }
  if (model_pos3) {
    if (ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "no model");
    memcpy(model_pos3, ctx->h_mpos.data(), (size_t)ctx->M * 12);
  }
  return STOCS_OK;
}

int stocs_b200_score_lcp_device(stocs_b200_ctx* ctx, const float* d_T16, int64_t H, float* d_lcp,
                                int32_t* d_inliers, void* stream) {
  if (!ctx) return STOCS_E_ARG;
  if (ctx->S <= 0 || ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "score_lcp: upload_model and upload_scene first");
  if (H < 0 || (H > 0 && (!d_T16 || !d_lcp))) STOCS_FAIL(ctx, STOCS_E_ARG, "score_lcp: bad argument");
  cudaSetDevice(ctx->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  ScoreRequest rq;
  rq.time_it = true;
  return stocs_launch_score(ctx, d_T16, H, d_lcp, d_inliers, st, rq);
}

int stocs_b200_score_lcp(stocs_b200_ctx* ctx, const float* T16, int64_t H, float* lcp, int32_t* inliers) {
  if (!ctx) return STOCS_E_ARG;
  if (ctx->S <= 0 || ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "score_lcp: upload_model and upload_scene first");
  if (H < 0 || (H > 0 && (!T16 || !lcp))) STOCS_FAIL(ctx, STOCS_E_ARG, "score_lcp: bad argument");
  if (H == 0) return STOCS_OK;
  cudaSetDevice(ctx->device);
  // the tail is the top-32 of the resident array, what stocs_b200_reduce_best(NULL) returns
  const int rc = stocs_score_host(ctx, "score_lcp", T16, H, lcp, inliers,
                                  [ctx, H](cudaStream_t st, const float*) { return enqueue_resident_topk(ctx, H, st); });
  ctx->top_valid = rc == STOCS_OK;
  return rc;
}

int stocs_b200_reduce_best_device(stocs_b200_ctx* ctx, const float* d_lcp, int64_t H, int K, int64_t index_offset,
                                  int64_t* d_topk_index, float* d_topk_lcp, void* stream) {
  if (!ctx) return STOCS_E_ARG;
  if (!d_lcp || H < 0 || !d_topk_index || !d_topk_lcp) STOCS_FAIL(ctx, STOCS_E_ARG, "reduce_best: bad argument");
  cudaSetDevice(ctx->device);
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  TopkRequest rq;
  rq.idx = d_topk_index;
  rq.val = d_topk_lcp;
  return stocs_launch_topk(ctx, d_lcp, H, K, index_offset, st, rq);
}

int stocs_b200_reduce_best(stocs_b200_ctx* ctx, const float* lcp, int64_t H, int K, int64_t* best_index,
                           float* best_lcp, int64_t* topk_index, float* topk_lcp) {
  if (!ctx) return STOCS_E_ARG;
  if (H < 0 || K < 1 || K > 32) STOCS_FAIL(ctx, STOCS_E_ARG, "reduce_best: bad argument");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  if (lcp) {
    ctx->top_valid = false;
    STOCS_CUDA(ctx, ctx->d_lcp.ensure((size_t)(H ? H : 1) * 4));
    if (H) STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->d_lcp.p, lcp, (size_t)H * 4, cudaMemcpyHostToDevice, st));
    ctx->last_H = H;
  } else if (ctx->last_H != H || !ctx->d_lcp.p) {
    STOCS_FAIL(ctx, STOCS_E_STATE, "reduce_best: no resident lcp array of that size");
  }
  // both branches reduce ctx->d_lcp; h_top may already hold its top-32 (score_lcp, an earlier call)
  if (!ctx->top_valid) {
    int rc = enqueue_resident_topk(ctx, H, st);
    if (rc) return rc;
    STOCS_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->top_valid = true;
  }
  // top-K is a prefix of top-32
  if (best_index) *best_index = ctx->h_top->idx[0];
  if (best_lcp) *best_lcp = ctx->h_top->val[0];
  for (int k = 0; k < K; ++k) {
    if (topk_index) topk_index[k] = ctx->h_top->idx[k];
    if (topk_lcp) topk_lcp[k] = ctx->h_top->val[k];
  }
  return STOCS_OK;
}

int stocs_b200_get_counters(stocs_b200_ctx* ctx, int64_t* counters, int n) {
  if (!ctx || !counters) return STOCS_E_ARG;
  cudaSetDevice(ctx->device);
  if (ctx->d_small.p) {
    DevScratch::ScoreTotals t{};
    STOCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    STOCS_CUDA(ctx, cudaMemcpy(&t, &ctx->scratch()->score_totals, sizeof(t), cudaMemcpyDeviceToHost));
    ctx->counters[CTR_TIES] = (int64_t)t.ties;
    ctx->counters[CTR_REJECTED_LOOP1] = (int64_t)t.rejected[0];
    ctx->counters[CTR_REJECTED_DRAIN] = (int64_t)t.rejected[1];
    ctx->counters[CTR_REJECTED_BRICK] = (int64_t)t.rejected[2];
  }
  for (int i = 0; i < n && i < CTR_COUNT; ++i) counters[i] = ctx->counters[i];
  return STOCS_OK;
}

// Data-dependent work of one scoring launch, counted by the counting variant of the kernel.
int stocs_b200_score_counters(stocs_b200_ctx* ctx, const float* d_T16, int64_t H, int64_t* counters, int n) {
  if (!ctx) return STOCS_E_ARG;
  if (ctx->S <= 0 || ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "score_counters: upload_model and upload_scene first");
  if (H <= 0 || !d_T16 || !counters || n < 1) STOCS_FAIL(ctx, STOCS_E_ARG, "score_counters: bad argument");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  DevBuf &d_lcp = ctx->pool[POOL_SHARD_LCP], &d_inl = ctx->pool[POOL_SHARD_INL];
  STOCS_CUDA(ctx, d_lcp.ensure((size_t)H * 4));
  STOCS_CUDA(ctx, d_inl.ensure((size_t)H * 4));
  unsigned long long* d_cnt = ctx->scratch()->score_counts;
  unsigned long long h[sizeof(DevScratch::score_counts) / 8] = {0};
  STOCS_CUDA(ctx, cudaMemsetAsync(d_cnt, 0, sizeof(h), st));
  ScoreRequest rq;
  rq.counters = d_cnt;
  int rc = stocs_launch_score(ctx, d_T16, H, d_lcp.as<float>(), d_inl.as<int32_t>(), st, rq);
  if (rc) return rc;
  STOCS_CUDA(ctx, cudaMemcpyAsync(h, d_cnt, sizeof(h), cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  int64_t out[9] = {H * (int64_t)ctx->M, (int64_t)h[0], (int64_t)h[1], (int64_t)h[2], (int64_t)h[3],
                    (int64_t)h[4], (int64_t)h[5], (int64_t)h[6], H};
  for (int i = 0; i < n && i < 9; ++i) counters[i] = out[i];
  return STOCS_OK;
}

int stocs_b200_kernel_ms_stats(stocs_b200_ctx* ctx, int reset, int32_t* n_launches, float* mean_ms, float* max_ms) {
  if (!ctx) return STOCS_E_ARG;
  cudaSetDevice(ctx->device);
  const int64_t n = ctx->ev_count < stocs_b200_ctx::kEvRing ? ctx->ev_count : stocs_b200_ctx::kEvRing;
  double sum = 0;
  float mx = 0.f;
  for (int64_t i = 0; i < n; ++i) {
    const int k = (int)((ctx->ev_count - 1 - i) % stocs_b200_ctx::kEvRing);
    float ms = 0.f;
    STOCS_CUDA(ctx, cudaEventSynchronize(ctx->ev_ring[2 * k + 1]));
    STOCS_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev_ring[2 * k], ctx->ev_ring[2 * k + 1]));
    sum += ms;
    if (ms > mx) mx = ms;
  }
  if (n_launches) *n_launches = (int32_t)n;
  if (mean_ms) *mean_ms = n ? (float)(sum / (double)n) : 0.f;
  if (max_ms) *max_ms = mx;
  if (reset) ctx->ev_count = 0;
  return STOCS_OK;
}

int stocs_b200_last_kernel_ms(stocs_b200_ctx* ctx, float* ms) {
  if (!ctx || !ms) return STOCS_E_ARG;
  if (!ctx->timing_valid || !ctx->ev0) STOCS_FAIL(ctx, STOCS_E_STATE, "no timed launch");
  cudaSetDevice(ctx->device);
  STOCS_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
  STOCS_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
  return STOCS_OK;
}

}  // extern "C"
