// stocs_ctx.h -- internal context shared by the translation units of libstocs_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <functional>
#include <string>
#include <vector>

#include "../../include/stocs_b200.h"
#include "stocs_math.h"

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  cudaError_t ensure(size_t need) {
    if (need <= bytes && p) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; bytes = 0;
    size_t cap = need < 256 ? 256 : need;
    cudaError_t e = cudaMalloc(&p, cap);
    if (e == cudaSuccess) bytes = cap;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
  template <class T> T* as() const { return (T*)p; }
};

// Device kd-tree node (16 B).  Inner: split/first/dim; leaf: start/size.
struct KdNodeDev {
  float split;
  uint32_t first_or_start;
  uint32_t dim_or_size;
  uint32_t leaf;
};

// Dense voxel grid over the centred scene with eps-dilated per-cell candidate lists.
struct GridDesc {
  float ox, oy, oz;   // origin (lower corner of cell 0)
  float inv_cell;     // 1 / cell edge
  int nx, ny, nz;
  int nbx, nby, nbz;  // bricks of 4x4x4 cells
  uint32_t nbricks;
  uint32_t ncells;    // nbricks * 64 (brick-major numbering)
};

// Parameters of a scene-index build between its enqueue and its completion (scene_index.cu)
struct IndexBuild {
  float r;                   // dilation radius of the candidate lists
  size_t cap;                // candidate records the buffers are sized for
  size_t nc1;                // cells + 1
  size_t tmp_bytes, tmp_bytes2;   // cub scratch of the two scans
};

struct PpfTableDesc {
  int n1, na;          // bins along the distance axis / each angle axis
  int tr, rot;
  int64_t npairs;      // ordered pairs stored (own bin)
  int64_t nkeys;       // occupied own bins
  int64_t nexpanded;   // keys of the reference's expanded map
};

// Scratch-pool slot names (stocs_b200_ctx::pool).  Ranges that overlap belong to stages that are
// never active inside the same ABI call on the same stream.
enum PoolSlot : int {
  // congruent.cu (stocs_congruent_enqueue): 0..11; POOL_CONG_QUADS is its output, read by run_pipeline
  POOL_CONG_INFO = 0, POOL_CONG_SEG, POOL_CONG_CODES_A, POOL_CONG_CODES_B, POOL_CONG_TMP, POOL_CONG_PE,
  POOL_CONG_QE, POOL_CONG_QCELL, POOL_CONG_CNT, POOL_CONG_SCAN, POOL_CONG_QOFF, POOL_CONG_QUADS = 11,
  // scene_index.cu (upload_scene): 12..15
  POOL_INDEX_DENSE = 12, POOL_INDEX_MASKS, POOL_INDEX_OCC, POOL_INDEX_OCC_SCAN,
  // scene_cloud.cu (build_scene_cloud[s]): 12..30; POOL_CLOUD_PROB holds one map per object, POOL_CLOUD_FLAGS
  // one row flag per (object, pixel)
  POOL_CLOUD_DEPTH = 12, POOL_CLOUD_BGR, POOL_CLOUD_PROB, POOL_CLOUD_EDGE, POOL_CLOUD_XYZ, POOL_CLOUD_KEYS_A,
  POOL_CLOUD_KEYS_B, POOL_CLOUD_IDX_A, POOL_CLOUD_IDX_B, POOL_CLOUD_TMP, POOL_CLOUD_FLAGS, POOL_CLOUD_SCAN,
  POOL_CLOUD_STARTS, POOL_CLOUD_UKEYS, POOL_CLOUD_CENT, POOL_CLOUD_KEEP, POOL_CLOUD_NRM, POOL_CLOUD_RC,
  POOL_CLOUD_OUT = 30,
  // ppf_table.cu (upload_model / upload_ppf_table): 16..18
  POOL_PPF_KEYS_A = 16, POOL_PPF_KEYS_B, POOL_PPF_CUB_TMP,
  // fit.cu (run_pipeline): 28..31
  POOL_PIPE_OFF = 28, POOL_PIPE_ITEMS, POOL_PIPE_FIT, POOL_PIPE_BASES = 31,
  // icp.cu: 32..36
  POOL_ICP_SRC = 32, POOL_ICP_TGT, POOL_ICP_TN, POOL_ICP_PART, POOL_ICP_STATE,
  // capi.cu: top-32 of the resident lcp array
  POOL_TOPK_RESIDENT = 37,
  // comm.cu: packed 64-byte records (local K, gathered world*K, merged K)
  POOL_COMM_SEND = 38, POOL_COMM_RECV, POOL_COMM_OUT,
  // sharded scoring scratch (transforms / lcp / inliers of the local shard)
  POOL_SHARD_T = 42, POOL_SHARD_LCP, POOL_SHARD_INL,
  // score.cu: claim order of the heavy-first schedule (one int per hypothesis of the launch), or of a
  // top-K launch in descending survivor count (one {hypothesis, count} uint2 per hypothesis)
  POOL_SCORE_ORDER = 45,
  // reduce.cu: per-CTA top-32 lists of reductions launched on the context's second stream
  POOL_TOPK_LISTS_AUX = 46,
  // congruent.cu / fit.cu: device scalars of one congruent-set search or pipeline run (StocsPipeState)
  POOL_PIPE_STATE = 47,
  // congruent.cu: bucket counters of the (base, cell) hash of the Q entries (zero between searches)
  POOL_CONG_HEAD = 48,
  // scene_index.cu: per-cell counters of the index build, zero between builds (state across calls by design)
  POOL_INDEX_COUNTS = 49,
  // congruent.cu: per-base table of cone directions
  POOL_CONG_CONE = 50,
  // congruent.cu: bucket number of every Q entry; bucket starts; {Q index, cell} records in bucket order
  POOL_CONG_NEXT = 51, POOL_CONG_BSTART = 52, POOL_CONG_BUCKET = 53,
  // score.cu: work counter, theta and bucket counts of a top-K-pruned scoring launch
  POOL_SCORE_PRUNE = 54,
  // cluster.cu: sort keys, cub scratch, kept poses (and the uploaded poses of stocs_b200_cluster_poses)
  POOL_CLUSTER = 55,
  // capi.cu (upload_scenes_device): a slice held on another device, copied to this one (pos3 | nrm3 | cls | pix)
  POOL_SCENE_PEER = 56,
  // score.cu: survivor count of every hypothesis of a top-K launch (survivor_count_kernel, fine map)
  POOL_SCORE_NS = 57,
  POOL_COUNT = 58
};

// Device scalars of one congruent-set search (congruent.cu) and of the pipeline run around it (fit.cu).
// Every list size of the online stages lives here, so the host enqueues the whole chain against
// CAPACITIES and reads this record back once at the end; a search that did not fit sets `overflow`
// (and turns its own later stages into no-ops), the host grows the buffers and enqueues it again.
struct StocsPipeState {
  unsigned long long need_codes;   // P + Q list entries of all bases (valid also when they did not fit)
  unsigned long long need_quads;   // congruent sets of all bases
  uint32_t totalP, total;          // entries of the flat code buffer in use: P lists first, then Q lists
  uint32_t total_quads;
  uint32_t overflow;               // 1: code buffers too small, 2: quad buffer too small, 4: pair lists >= 2^28 entries
  long long n_items;               // transforms to fit (at most max_sets per base)
  long long n_ok;                  // of which pass the fit's orthogonality test
  long long best_item, rank_of_best;
  int n_valid, best_base;
  float best_lcp;
  int n_poses;                     // poses kept by the clustering of a clustered run (cluster.cu)
  float best_Tc[16], best_Tw[16];
};

// Slots of stocs_b200_ctx::counters.  [0]-[5] and [8] are public: stocs_b200_get_counters returns
// them, and include/stocs_b200.h documents what they count.  [6] and [7] are internal.
enum CtxCounter : int {
  CTR_SCORE_LAUNCHES = 0,   // score kernels launched (icp.cu adds the launches of its iterations)
  CTR_TIES,                 // NN queries resolved by the kd-tree tie path (DevScratch::score_totals)
  CTR_GRID_CELLS,           // grid cells of the current scene index
  CTR_CANDIDATES,           // replicated candidate records of the current scene index
  CTR_REJECTED_LOOP1,       // top-K hypotheses rejected on the prefilter count: fine-map survivor count or loop 1 (DevScratch::score_totals)
  CTR_REJECTED_DRAIN,       // top-K hypotheses rejected before a queue drain (DevScratch::score_totals)
  CTR_OCCUPIED_CELLS,       // occupied cells of the current scene index
  // STATE, not a diagnostic: voxels of the last build_scene_cloud, which the next call takes as its
  // guess of how many points to read back in the same queue as the list lengths (scene_cloud.cu)
  CTR_CLOUD_VOXELS,
  CTR_REJECTED_BRICK,       // top-K hypotheses rejected after the brick-bit refinement (DevScratch::score_totals)
  CTR_COUNT
};

struct DevScratch;

// What the device tells the host about a scene in device memory before its index is laid out
// (stocs_index_centre_device): one 64-byte record, reduced in DevScratch::plan and copied to ctx->h_plan.
struct ScenePlan {
  float centroid[4];
  int aabb[6];                  // box of the centred points as ordered ints (min xyz, max xyz)
  int wbits;                    // bits of the largest class weight before first_bad
  int first_bad;                // first class weight that is negative, NaN or infinite; INT_MAX: none
  int pix_min[2], pix_max[2];   // (row, col) range; min > max: no pixel coordinates
};
static_assert(sizeof(ScenePlan) == 64, "ScenePlan is one 64-byte read-back");

struct stocs_b200_ctx {
  int device = 0;
  int num_sms = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;
  cudaStream_t aux_stream = nullptr;   // second compute stream: consecutive score chunks overlap their tails
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // the most recent timed scoring launch (aliases into ev_ring)
  // ring of event pairs around the timed scoring launches (stocs_b200_kernel_ms_stats)
  static constexpr int kEvRing = 512;
  cudaEvent_t ev_ring[2 * kEvRing] = {};
  int64_t ev_count = 0;
  static constexpr int kMaxChunks = 4;    // chunks of the staged host-buffer scoring plan (stocs_score_host)
  cudaEvent_t chunk_ev[kMaxChunks] = {};  // H2D-complete events of those chunks
  cudaEvent_t join_ev[2] = {nullptr, nullptr};
  std::string err;

  // parameters
  float eps = 0.005f;
  int tr = 5, rot = 5;
  float dot_thr = 0.f;  // "angle < 30" <=> dot_thr < dot <= 1 (see angle_threshold_dot)

  // model (centred)
  int M = 0, Mpad = 0;
  float model_abs_max = 0.f;           // largest |coordinate| of the centred model (NaN if one is not finite)
  float cm[3] = {0, 0, 0};
  std::vector<float> h_mpos, h_mnrm;  // centred positions, normals (M*3)
  DevBuf d_model;                      // 8*Mpad floats: float4 positions, then float4 normals
  DevBuf d_mpos4;                      // float4 (x,y,z,0) centred
  DevBuf d_mnrm4;                      // float4 (nx,ny,nz,0)

  // scene (centred)
  int S = 0;
  int S_pending = 0;                   // size of the scene being uploaded (S is committed on success)
  const float* h_pos_pending = nullptr;  // its positions in the caller's host buffer (valid during upload_scene only)
  bool scene_empty = false;            // S == 0 because upload_scenes gave this context an empty slice
  IndexBuild index_build{};            // the index build in flight (stocs_index_enqueue -> stocs_index_complete)
  float h_centroid_stage[4] = {0, 0, 0, 0};  // source of the 12-byte centroid upload (must outlive the async copy)
  float cs[3] = {0, 0, 0};
  std::vector<float> h_spos;           // centred positions (S*3) of a scene from host memory: the kd-tree thread's input
  bool plan_on_device = false;         // the scene is planned on the device (between stocs_index_plan and _finish)
  DevBuf d_spos4;                      // float4 (x,y,z,bits(idx))
  DevBuf d_sattr;                      // float4 (nx,ny,nz,class probability)
  DevBuf d_spix;                       // int2 (row, col)
  bool has_pixels = false;
  int pix_min[2] = {0, 0}, pix_max[2] = {0, 0};  // (row, col) range of the uploaded pixel coordinates
  // instance-mode state (edge map, previous_segment | segmentation_buffer | current mask, cached masks)
  DevBuf d_edge, d_inst_state, d_mask_store, d_frontier;
  int img_w = 0, img_h = 0;
  GridDesc grid{};
  float w_max = 0.f;                   // largest class weight of the scene (top-K pruning bound, score.cu)
  bool prune_ok = false;               // every class weight finite and >= 0: top-K pruning allowed
  DevBuf d_brick_occ;                  // 1 bit per brick: brick has an occupied cell
  DevBuf d_coarse;                     // 1 bit per block of 2^coarse_shift cells/axis (>= brick): block has an occupied cell
  int coarse_shift = 2, coarse_nx = 0, coarse_ny = 0, coarse_nz = 0, coarse_words = 0;
  // the same map at blocks of 2^fine_shift cells/axis (2 <= fine_shift <= coarse_shift), for the top-K
  // survivor count only; fine_shift == coarse_shift: no second map, d_fine is unused and the count reads d_coarse
  DevBuf d_fine;
  int fine_shift = 2, fine_nx = 0, fine_ny = 0, fine_nz = 0, fine_words = 0;
  DevBuf d_bricks;                    // uint4 {mask lo, mask hi, first occupied-cell rank, 0} per brick
  DevBuf d_cell_start;                 // uint32[occupied cells + 1]: candidate offsets
  DevBuf d_cand;                       // float4 (x,y,z,bits(idx)) replicated per dilated cell
  int64_t ncand = 0;
  DevBuf d_kd_nodes, d_kd_pts;         // reference kd-tree for exact-tie resolution
  DevBuf d_kd_build;                   // scratch of its device build (in use until kd_copy_done, across calls)
  int kd_nodes = 0;

  // PPF table
  PpfTableDesc ppf{};
  DevBuf d_ppf_bin_start;              // uint32[nbins+1]  CSR over own bins
  DevBuf d_ppf_pairs;                  // uint32 (id1<<16|id2) sorted by (bin, id1, id2)
  DevBuf d_ppf_keybits;                // bitmap of keys present in the reference's expanded map
  std::vector<uint32_t> h_ppf_bin_start, h_ppf_pairs;

  // grow-only scratch slots reused by the multi-kernel stages (no cudaMalloc/cudaFree per call).
  // Slots are named by PoolSlot below.  Rule: a slot is single-stream scratch -- no slot may hold
  // state across ABI calls, so stages that never run inside one another may share a number.  Two
  // deliberate exceptions, each with a number of its own: POOL_INDEX_COUNTS and POOL_CONG_HEAD are
  // counter arrays that every run leaves ZEROED (tracked by index_counts_clean / cong_bcount_clean),
  // so that the next run need not clear tens of megabytes first.
  DevBuf pool[POOL_COUNT];
  // scratch (d_small: 4 KB, laid out by DevScratch)
  DevBuf d_T, d_lcp, d_inl, d_work, d_tmp, d_tmp2, d_small;
  DevScratch* scratch() const { return d_small.as<DevScratch>(); }

  // capacities the online stages are enqueued against (entries; grown when a search reports overflow)
  long long cong_cap_codes = 1 << 18, cong_cap_quads = 1 << 21;
  long long cong_table_size = 0;       // buckets the counters in pool[POOL_CONG_HEAD] were cleared for
  bool cong_bcount_clean = false;      // ... and whether the last search left them zero
  long long pipe_last_items = 0;       // transforms of the previous pipeline run (sizes the next run's grids)
  StocsPipeState* h_pipe_state = nullptr;   // page-locked landing zone of the state record
  struct ClusterHost* h_cluster = nullptr;  // page-locked landing zone of the clustering results (cluster.cu)
  uint32_t* h_index_counts = nullptr;       // page-locked: list lengths of the scene-index build [0, 8) and of
                                            // the scene-cloud build [8, 8 + 1 + STOCS_B200_MAX_CLOUD_OBJECTS)
  size_t index_counts_clean = 0;            // leading words of pool[POOL_INDEX_COUNTS] known to be zero
  void* h_kd_stage = nullptr;               // page-locked staging of the kd-tree upload (frame-sized scenes)
  size_t h_kd_stage_bytes = 0;
  ScenePlan* h_plan = nullptr;              // page-locked landing zone of a device plan's record
  struct KdPending* kd_pending = nullptr;   // kd-tree of the current scene, still being built (host thread or device)
  cudaEvent_t kd_copy_done = nullptr;       // the staging buffer may be overwritten / the device build is complete

  // resident lcp array (d_lcp / d_inl) of the last host-buffer score call or explicit reduce_best
  int64_t last_H = 0;
  // top-32 of the resident lcp array, computed by score_lcp behind its result copies and by reduce_best
  struct TopCache { int64_t idx[32]; float val[32]; };
  TopCache* h_top = nullptr;   // page-locked
  bool top_valid = false;
  int64_t counters[CTR_COUNT] = {0};
  // points of the last build_scene_cloud[s] (all objects): with CTR_CLOUD_VOXELS, the next call's read-back estimate
  long long cloud_last_points = 0;
  bool timing_valid = false;

  // multi-GPU (comm.cu): one NCCL communicator per context; ncclComm_t kept opaque here
  void* comm = nullptr;
  int comm_rank = 0, comm_nranks = 1;
};

// Small device values of the stages, in the context's 4 KB scratch (stocs_b200_ctx::d_small).
// stocs_b200_create zeroes it once.  Fields marked ZERO-RELIANT count on that and are never cleared
// again; every other field is written by its stage before it is read.
struct DevScratch {
  // score.cu: work counter of a scoring launch per slot (slot 0 by default, staged host-buffer chunks use
  // their chunk number so that concurrent chunks do not share one); cleared before each launch
  unsigned long long work[stocs_b200_ctx::kMaxChunks];
  // score.cu, ZERO-RELIANT: NN queries resolved by the kd-tree tie path, and top-K hypotheses
  // rejected on the prefilter count / before a drain / after the brick-bit refinement, accumulated
  // over the context's lifetime; stocs_b200_get_counters reads the four in one copy
  struct ScoreTotals { unsigned long long ties, rejected[3]; } score_totals;
  // capi.cu (stocs_b200_score_counters): the counting variant's ScoreCounter slots (score.cu)
  unsigned long long score_counts[8];
  // reduce.cu, ZERO-RELIANT: top-K ticket of the context stream [0] and of its second stream [1];
  // the last CTA of a launch resets it
  unsigned topk_ticket[2];
  // score.cu: heavy-first schedule, next position from the front (heavy) and from the back (light)
  unsigned lpt_fill[2];
  // score.cu (stocs_fmad_selftest): written after the creation memset, so shared with no other field
  float fmad_selftest;
  // scene_index.cu: centroid of stocs_centre_points; the device plan of a scene (stocs_index_centre_device)
  ScenePlan plan;
  // ppf_table.cu: occupied keys of the table build, entries of a lookup, entries an upload rejected
  unsigned long long ppf_nkeys;
  long long ppf_lookup_n;
  unsigned long long ppf_bad;
  // fit.cu: best transform of the pipeline's top-1 reduction (index, lcp)
  long long pipe_best_idx;
  float pipe_best_lcp;
  // sample_instance.cu (stocs_b200_sample_instance_base): base point ids, inverse distances, valid flag
  int inst_ids[4];
  float inst_inv[2];
  uint8_t inst_valid;
  // scene_cloud.cu (build_scene_clouds): first zero-depth pixel, zero-depth pixels, valid pixels, voxels, then
  // the end of each object's rows in the concatenated output
  int cloud[4 + STOCS_B200_MAX_CLOUD_OBJECTS];
};
static_assert(sizeof(DevScratch) <= 4096, "DevScratch must fit the 4 KB d_small allocation");

#define STOCS_CUDA(ctx, call)                                                            \
  do {                                                                                   \
    cudaError_t _e = (call);                                                             \
    if (_e != cudaSuccess) {                                                             \
      (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(_e);                   \
      return STOCS_E_CUDA;                                                               \
    }                                                                                    \
  } while (0)

#define STOCS_FAIL(ctx, code, msg) \
  do { (ctx)->err = (msg); return (code); } while (0)

// kernels / stages implemented in the other translation units
// scene index of ctx->S_pending points (scene_index.cu), in three steps: plan (grow every buffer; for a scene
// in host memory also centre on the host, start the kd-tree thread and lay out the grid; nothing enqueued),
// enqueue (device centring of host positions in ctx->d_tmp or the device kd-tree build, the index kernels and
// their two length copies), complete (wait, grow and run again if the candidate records did not fit, commit
// the counters).  A scene in device memory is planned between the first two: centre_device enqueues the
// centring and the plan record's copy, plan_finish waits for it and lays out the grid.
int stocs_index_plan(stocs_b200_ctx* ctx);
int stocs_index_centre_device(stocs_b200_ctx* ctx, const float* d_pos3, const float* d_cls, const int32_t* d_pix);
int stocs_index_plan_finish(stocs_b200_ctx* ctx);
int stocs_index_enqueue(stocs_b200_ctx* ctx);
int stocs_index_complete(stocs_b200_ctx* ctx);
// reference centroid of n host points (h_pos3) into h_centroid3, their centred copy into h_centred3, and the
// same centring on the device of their copy d_pos3 into d_out4 (enqueued, no synchronisation)
int stocs_centre_points(stocs_b200_ctx* ctx, const float* d_pos3, int n, float4* d_out4, float* h_centroid3,
                        const float* h_pos3, float* h_centred3);
int stocs_pack_scene_attr(stocs_b200_ctx* ctx, const float* d_nrm3, const float* d_cls, int S);
// One scoring launch (score.cu).  The caller states which instantiation it wants: per-hypothesis
// results (the default), only the K best (top_K = K: hypotheses that provably cannot enter them may
// be left unscored, lcp 0, see kPrune; slot 0 only, no device count) or counting (counters: the
// ScoreCounter slots).
struct ScoreRequest {
  bool time_it = false;                    // events around the launch (stocs_b200_kernel_ms_stats)
  int slot = 0;                            // work counter; launches that may run concurrently take distinct slots
  int top_K = 0;
  unsigned long long* counters = nullptr;
  const long long* d_H = nullptr;          // the count lives on the device, H bounds it ...
  long long grid_hint = 0;                 // ... and grid_hint sizes the launch
};
int stocs_launch_score(stocs_b200_ctx* ctx, const float* d_T, int64_t H, float* d_lcp, int32_t* d_inl,
                       cudaStream_t st, const ScoreRequest& rq);
// survivor count of each of H device transforms into d_ns (score.cu; enqueued on st, lcp written to
// scratch): on the fine map as a large top-K launch orders its claims by it (fine), or on the coarse map
// as loop 1 counts (!fine)
int stocs_survivor_counts(stocs_b200_ctx* ctx, const float* d_T, int64_t H, unsigned* d_ns, cudaStream_t st, bool fine);
int stocs_launch_backproject(stocs_b200_ctx* ctx, const uint16_t* d_depth, const uint8_t* d_bgr,
                             int W, int H, float fx, float cx, float fy, float cy, float scale,
                             float* d_xyz, uint32_t* d_rgb, cudaStream_t st);  // backproject.cu
// joins the kd-tree build started by upload_scene (if any) and, with upload = true, queues its upload on st
int stocs_kd_finish(stocs_b200_ctx* ctx, cudaStream_t st, bool upload = true);  // scene_index.cu
bool stocs_fmad_selftest(stocs_b200_ctx* ctx);                             // score.cu
// device alias of page-locked host memory, NULL for any other pointer (capi.cu)
const void* stocs_host_alias(const void* p);
// p is device memory (cudaMalloc'd or managed) on `device`, or on any device when device < 0; its device goes to
// *owner (capi.cu)
bool stocs_device_memory(const void* p, int device, int* owner = nullptr);
// The calls that read a caller's device buffers order their work after what the caller has queued on its stream
// so far: an event recorded there (a stream of `device`; NULL is that device's default stream, as everywhere in
// CUDA, and torch's default stream), which context streams wait for.
struct CallerEvent {
  cudaEvent_t ev = nullptr;
  cudaError_t record(void* stream, int device) {
    int cur = 0;
    cudaError_t e = cudaGetDevice(&cur);
    if (e == cudaSuccess) e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventRecord(ev, stream ? (cudaStream_t)stream : cudaStreamLegacy);
    cudaSetDevice(cur);
    return e;
  }
  cudaError_t wait(cudaStream_t st) const { return cudaStreamWaitEvent(st, ev, 0); }
  CallerEvent() = default;
  CallerEvent(const CallerEvent&) = delete;
  CallerEvent& operator=(const CallerEvent&) = delete;
  ~CallerEvent() { if (ev) cudaEventDestroy(ev); }   // released once recorded work completes
};
// device alias through which a host-buffer scoring call reads its transforms in place, NULL when
// they are staged instead: pageable memory, or STOCS_NO_ZERO_COPY set (capi.cu)
const float* stocs_zero_copy_transforms(const float* T16);
// w_max / prune_ok of the scene from its class weights (capi.cu; every writer of the weights calls it)
void stocs_set_weight_bound(stocs_b200_ctx* ctx, const float* cls, int S);
// Outputs of one top-K reduction of a device lcp array (reduce.cu): the K best as (index, lcp)
// pairs (idx and val together) and/or as 64-byte records, which read the scored transforms (T16)
// and inlier counts (inl, may be NULL) as well
struct TopkRequest {
  int64_t* idx = nullptr;
  float* val = nullptr;
  const float* T16 = nullptr;
  const int32_t* inl = nullptr;
  stocs_b200_record* rec = nullptr;
  const long long* d_H = nullptr;          // as for ScoreRequest
  long long grid_hint = 0;
};
int stocs_launch_topk(stocs_b200_ctx* ctx, const float* d_lcp, int64_t H, int K, int64_t index_offset,
                      cudaStream_t st, const TopkRequest& rq);
// Host-buffer scoring (capi.cu; stocs_b200_score_lcp, stocs_b200_score_sharded): scores H host
// transforms into the resident ctx->d_lcp / d_inl, copies back whichever of lcp / inliers is
// non-NULL, enqueues tail(stream, device-visible transforms), joins the second stream and
// synchronises once.  After the first error nothing more is enqueued, but the join and the
// synchronisation still happen; that first error is returned.  On success the resident array
// holds H results (last_H); on failure last_H is 0.  H == 0: nothing is scored, the resident
// state is untouched and only the tail runs, on the context stream.  `who` prefixes error messages.
using ScoreTail = std::function<int(cudaStream_t, const float*)>;
int stocs_score_host(stocs_b200_ctx* ctx, const char* who, const float* T16, int64_t H, float* lcp, int32_t* inliers,
                     const ScoreTail& tail);
float stocs_angle_threshold_dot();                                         // capi.cu (host)
// Greedy clustering of a pipeline run's scored list (cluster.cu), enqueued behind pipe_finalize_kernel:
// candidates are the fitted items (ok) below the device count, best score = the state's best_lcp; the
// kept poses land in ctx->h_cluster and their number in the state record's n_poses.
struct PipeClusterInputs {
  const float* lcp; const float* Tc; const float* Tw;
  const uint8_t* ok; const uint8_t* valid; const int* item_base;
  long long cap_items;
  StocsPipeState* d_state;
};
int stocs_cluster_check(stocs_b200_ctx* ctx, const stocs_b200_cluster_params* p, int64_t cap);
// Calls over one context per object (capi.cu): stocs_batch_check rejects n_objects < 1, a NULL entry and
// a context given twice; stocs_batch_fail sets "who: object k: msg" on ctxs[k] and ctxs[0] (k < 0: on
// ctxs[0] only, without an object) and returns code.
int stocs_batch_check(stocs_b200_ctx* const* ctxs, int n_objects, const char* who);
int stocs_batch_fail(stocs_b200_ctx* const* ctxs, int k, int code, const char* who, const std::string& msg);
// the context can run instance-mode sampling: edge map, pixel coordinates inside it (sample_instance.cu)
int stocs_instance_check(stocs_b200_ctx* ctx);
int stocs_cluster_enqueue_pipeline(stocs_b200_ctx* ctx, const stocs_b200_cluster_params& p, const PipeClusterInputs& in,
                                   cudaStream_t st);
// grows the scratch of stocs_cluster_enqueue_pipeline over cap_items items; enqueues nothing
int stocs_cluster_reserve(stocs_b200_ctx* ctx, long long cap_items);
const stocs_b200_pose* stocs_cluster_poses_host(stocs_b200_ctx* ctx);
void stocs_cluster_free_host(stocs_b200_ctx* ctx);

// STOCS_TRACE=1: wall-clock of each stage of a host-driven sequence on stderr (adds a synchronize
// per stage, so the total is not the untraced time).
struct StageTrace {
  bool on; cudaStream_t st; std::chrono::steady_clock::time_point t0;
  explicit StageTrace(cudaStream_t s) : on(getenv("STOCS_TRACE") != nullptr), st(s), t0(std::chrono::steady_clock::now()) {}
  void mark(const char* what) {
    if (!on) return;
    cudaStreamSynchronize(st);
    const auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[stocs trace] %-28s %8.1f us\n", what, std::chrono::duration<double, std::micro>(t1 - t0).count());
    t0 = t1;
  }
};
