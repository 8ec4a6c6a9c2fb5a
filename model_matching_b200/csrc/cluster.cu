// cluster.cu -- clustering::greedy_clustering (reference src/pose_clustering.cpp:79-122) on the device.
//
// Filter and order come from reduce.cu's keys: (ordered lcp bits << 32) | ~index, sorted descending
// by cub, so the walk order is lcp descending with the lower index first among equal lcps (the shim's
// std::stable_sort) and every non-candidate (key 0) sorts behind the candidates.  The greedy walk is
// inherently sequential -- a candidate's fate depends on every pose kept before it -- and runs in ONE
// CTA: the sorted list is read in tiles of kThreads; each thread tests its candidate against the poses
// kept so far (in shared memory), then the tile is settled in order: its first survivor is kept, the
// later survivors are tested against that pose, and so on.  The translation test decides before the
// rotation is evaluated: the suppression condition is an AND, so this cannot change a decision.
// The pose distance is csrc/stocs_pose_math.h, the statement the host shim's get_pose_diff calls.
#include <cstring>

#include "stocs_ctx.h"
#include "stocs_pose_math.h"

using namespace stocsm;

int stocs_enqueue_cluster_keys(stocs_b200_ctx* ctx, const float* d_lcp, int64_t H, float thr, const float* d_thr_scale,
                               const uint8_t* d_ok, const long long* d_H, unsigned long long* keys,
                               unsigned long long* keys_out, void* tmp, size_t* tmp_bytes, cudaStream_t st);  // reduce.cu

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxPoses = 1024;   // maximum_pose_count + 1 kept poses live in shared memory (64 KB)

struct ClusterDevParams {
  float min_distance, min_angle;
  float sym[3];
  int max_count;
};

// does kept pose c suppress the candidate (T, ti = its inverse rotation)?
// get_pose_diff(candidate, c): rotation < min_angle && translation < min_distance
__device__ __forceinline__ bool suppressed_by(const float* T, const float ti[3][3], const float* c, const ClusterDevParams& p) {
  if (!(pose_translation_error(T, c) < p.min_distance)) return false;
  return pose_rotation_error(ti, c, p.sym) < p.min_angle;
}

// One CTA.  keys: H sorted keys (candidates first); Tw: the poses, 16 floats each, indexed by the key's
// index.  kept[0..*n_kept): the indices of the kept poses in the order they were kept.
__global__ void __launch_bounds__(kThreads) greedy_cluster_kernel(const unsigned long long* __restrict__ keys, long long H,
                                                                 const float* __restrict__ Tw, ClusterDevParams p,
                                                                 long long* __restrict__ kept, int* __restrict__ n_kept) {
  extern __shared__ float s_pose[];   // kept poses, 16 floats each
  __shared__ unsigned s_mask[kWarps];
  __shared__ int s_n;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  if (t == 0) s_n = 0;
  __syncthreads();
  bool done = false;
  for (long long tile = 0; tile < H && !done; tile += kThreads) {
    const long long pos = tile + t;
    const unsigned long long key = pos < H ? keys[pos] : 0ull;
    bool alive = key != 0ull;
    long long item = -1;
    float T[16], ti[3][3];
    if (alive) {
      item = (long long)(0xffffffffull - (key & 0xffffffffull));
#pragma unroll
      for (int k = 0; k < 16; ++k) T[k] = Tw[16 * item + k];
      pose_test_inverse(T, ti);
      const int n = s_n;
      for (int c = 0; c < n && alive; ++c) alive = !suppressed_by(T, ti, s_pose + 16 * c, p);
    }
    // settle the tile in order
    for (;;) {
      const unsigned m = __ballot_sync(0xffffffffu, alive);
      if (lane == 0) s_mask[w] = m;
      __syncthreads();
      int first = -1;
      for (int k = 0; k < kWarps; ++k) {
        const unsigned mk = s_mask[k];
        if (mk) { first = k * 32 + __ffs(mk) - 1; break; }
      }
      const int c = s_n;
      __syncthreads();
      if (first < 0) break;
      if (t == first) {
#pragma unroll
        for (int k = 0; k < 16; ++k) s_pose[16 * c + k] = T[k];
        kept[c] = item;
        s_n = c + 1;
        alive = false;
      }
      __syncthreads();
      if (c + 1 > p.max_count) { done = true; break; }   // the reference's break: more than maximum_pose_count kept
      if (alive) alive = !suppressed_by(T, ti, s_pose + 16 * c, p);
    }
    // candidates end at the first key 0 (the list is sorted); this is also the barrier before the next tile
    if (__syncthreads_or(key == 0ull)) break;
  }
  __syncthreads();
  if (t == 0) *n_kept = s_n;
}

// pipeline records (one block per kept pose): the index is the rank among the fitted items, the base
// the rank among the valid bases (PoseCandidate::base_index), as pipe_finalize_kernel ranks the best pose
__global__ void __launch_bounds__(256) cluster_records_kernel(const long long* __restrict__ kept, const int* __restrict__ n_kept,
                                                              const float* __restrict__ lcp, const uint8_t* __restrict__ ok,
                                                              const uint8_t* __restrict__ valid, const int* __restrict__ item_base,
                                                              const float* __restrict__ Tc, const float* __restrict__ Tw,
                                                              stocs_b200_pose* __restrict__ out) {
  __shared__ long long s_ok[8];
  __shared__ int s_valid[8];
  const int b = blockIdx.x;
  if (b >= *n_kept) return;
  const long long item = kept[b];
  const int base = item_base[item];
  long long n_ok = 0;
  int n_valid = 0;
  for (long long i = threadIdx.x; i < item; i += blockDim.x) n_ok += ok[i] ? 1 : 0;
  for (int k = threadIdx.x; k < base; k += blockDim.x) n_valid += valid[k] ? 1 : 0;
  for (int o = 16; o > 0; o >>= 1) {
    n_ok += __shfl_xor_sync(0xffffffffu, n_ok, o);
    n_valid += __shfl_xor_sync(0xffffffffu, n_valid, o);
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { s_ok[w] = n_ok; s_valid[w] = n_valid; }
  __syncthreads();
  stocs_b200_pose& r = out[b];
  if (threadIdx.x == 0) {
    for (int k = 1; k < 8; ++k) { n_ok += s_ok[k]; n_valid += s_valid[k]; }
    r.index = n_ok;
    r.lcp = lcp[item];
    r.base = n_valid;
  }
  if (threadIdx.x < 16) r.T_centred[threadIdx.x] = Tc[16 * item + threadIdx.x];
  else if (threadIdx.x < 32) r.T_world[threadIdx.x - 16] = Tw[16 * item + threadIdx.x - 16];
}

}  // namespace

// page-locked landing zone: the count and kept indices of cluster_poses, the records of a clustered run
struct ClusterHost {
  int n;
  long long kept[kMaxPoses];
  stocs_b200_pose poses[kMaxPoses];
};

namespace {

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// POOL_CLUSTER: [kept indices | count | records | keys | sorted keys | cub scratch | poses | lcps]
struct ClusterScratch {
  long long* kept; int* n; stocs_b200_pose* rec;
  unsigned long long* keys; unsigned long long* keys_sorted;
  void* tmp; size_t tmp_bytes;
  float* T; float* lcp;
};

int cluster_scratch(stocs_b200_ctx* ctx, long long H, bool host_inputs, cudaStream_t st, ClusterScratch& s) {
  s.tmp_bytes = 0;
  int rc = stocs_enqueue_cluster_keys(ctx, nullptr, H, 0.f, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, &s.tmp_bytes, st);
  if (rc) return rc;
  const size_t o_n = align256(kMaxPoses * 8), o_rec = o_n + 256, o_keys = o_rec + align256(kMaxPoses * sizeof(stocs_b200_pose));
  const size_t o_sorted = o_keys + align256((size_t)H * 8), o_tmp = o_sorted + align256((size_t)H * 8);
  const size_t o_T = o_tmp + align256(s.tmp_bytes), o_lcp = o_T + (host_inputs ? align256((size_t)H * 64) : 0);
  const size_t total = o_lcp + (host_inputs ? align256((size_t)H * 4) : 0);
  DevBuf& buf = ctx->pool[POOL_CLUSTER];
  STOCS_CUDA(ctx, buf.ensure(total));
  char* p = buf.as<char>();
  s.kept = (long long*)p; s.n = (int*)(p + o_n); s.rec = (stocs_b200_pose*)(p + o_rec);
  s.keys = (unsigned long long*)(p + o_keys); s.keys_sorted = (unsigned long long*)(p + o_sorted); s.tmp = p + o_tmp;
  s.T = host_inputs ? (float*)(p + o_T) : nullptr;
  s.lcp = host_inputs ? (float*)(p + o_lcp) : nullptr;
  if (!ctx->h_cluster) STOCS_CUDA(ctx, cudaHostAlloc((void**)&ctx->h_cluster, sizeof(ClusterHost), cudaHostAllocDefault));
  return STOCS_OK;
}

int enqueue_greedy(stocs_b200_ctx* ctx, const stocs_b200_cluster_params& p, const ClusterScratch& s, long long H,
                   const float* d_Tw, int* d_n, cudaStream_t st) {
  ClusterDevParams dp;
  dp.min_distance = p.min_distance; dp.min_angle = p.min_angle;
  for (int k = 0; k < 3; ++k) dp.sym[k] = p.sym_info[k];
  dp.max_count = p.maximum_pose_count;
  const int smem = (p.maximum_pose_count + 1) * 64;
  STOCS_CUDA(ctx, cudaFuncSetAttribute(greedy_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxPoses * 64));
  greedy_cluster_kernel<<<1, kThreads, smem, st>>>(s.keys_sorted, H, d_Tw, dp, s.kept, d_n);
  STOCS_CUDA(ctx, cudaGetLastError());
  return STOCS_OK;
}

}  // namespace

int stocs_cluster_check(stocs_b200_ctx* ctx, const stocs_b200_cluster_params* p, int64_t cap) {
  if (!p) STOCS_FAIL(ctx, STOCS_E_ARG, "cluster: params are NULL");
  if (p->maximum_pose_count < 0 || p->maximum_pose_count >= kMaxPoses)
    STOCS_FAIL(ctx, STOCS_E_ARG, "cluster: maximum_pose_count must be in 0..1023");
  if (cap < (int64_t)p->maximum_pose_count + 1) STOCS_FAIL(ctx, STOCS_E_ARG, "cluster: capacity below maximum_pose_count + 1");
  return STOCS_OK;
}

int stocs_cluster_enqueue_pipeline(stocs_b200_ctx* ctx, const stocs_b200_cluster_params& p, const PipeClusterInputs& in,
                                   cudaStream_t st) {
  if (in.cap_items >= (1ll << 31)) STOCS_FAIL(ctx, STOCS_E_ARG, "run_pipeline_clustered: more than 2^31 transforms");
  ClusterScratch s;
  int rc = cluster_scratch(ctx, in.cap_items, false, st, s);
  if (rc) return rc;
  rc = stocs_enqueue_cluster_keys(ctx, in.lcp, in.cap_items, p.acceptable_fraction, &in.d_state->best_lcp, in.ok,
                                  &in.d_state->n_items, s.keys, s.keys_sorted, s.tmp, &s.tmp_bytes, st);
  if (rc) return rc;
  rc = enqueue_greedy(ctx, p, s, in.cap_items, in.Tw, &in.d_state->n_poses, st);
  if (rc) return rc;
  const int nrec = p.maximum_pose_count + 1;
  cluster_records_kernel<<<nrec, 256, 0, st>>>(s.kept, &in.d_state->n_poses, in.lcp, in.ok, in.valid, in.item_base, in.Tc,
                                               in.Tw, s.rec);
  STOCS_CUDA(ctx, cudaGetLastError());
  STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->h_cluster->poses, s.rec, (size_t)nrec * sizeof(stocs_b200_pose), cudaMemcpyDeviceToHost, st));
  return STOCS_OK;
}

int stocs_cluster_reserve(stocs_b200_ctx* ctx, long long cap_items) {
  ClusterScratch s;
  return cluster_scratch(ctx, cap_items, false, ctx->stream, s);
}

const stocs_b200_pose* stocs_cluster_poses_host(stocs_b200_ctx* ctx) { return ctx->h_cluster->poses; }

void stocs_cluster_free_host(stocs_b200_ctx* ctx) {
  if (ctx->h_cluster) cudaFreeHost(ctx->h_cluster);
  ctx->h_cluster = nullptr;
}

extern "C" int stocs_b200_cluster_poses(stocs_b200_ctx* ctx, const float* T16_world, const float* lcp, int64_t H,
                                        float best_score, const stocs_b200_cluster_params* p,
                                        int64_t* index_out, int64_t cap, int64_t* n_out) {
  if (!ctx) return STOCS_E_ARG;
  int rc = stocs_cluster_check(ctx, p, cap);
  if (rc) return rc;
  if (!n_out || !index_out || H < 0 || H >= (1ll << 31) || (H > 0 && (!T16_world || !lcp)))
    STOCS_FAIL(ctx, STOCS_E_ARG, "cluster_poses: bad argument");
  *n_out = 0;
  if (H == 0) return STOCS_OK;
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  ClusterScratch s;
  rc = cluster_scratch(ctx, H, true, st, s);
  if (rc) return rc;
  STOCS_CUDA(ctx, cudaMemcpyAsync(s.T, T16_world, (size_t)H * 64, cudaMemcpyHostToDevice, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(s.lcp, lcp, (size_t)H * 4, cudaMemcpyHostToDevice, st));
  const float thr = p->acceptable_fraction * best_score;   // binary32, as the reference's filter
  rc = stocs_enqueue_cluster_keys(ctx, s.lcp, H, thr, nullptr, nullptr, nullptr, s.keys, s.keys_sorted, s.tmp, &s.tmp_bytes, st);
  if (rc) return rc;
  rc = enqueue_greedy(ctx, *p, s, H, s.T, s.n, st);
  if (rc) return rc;
  ClusterHost* h = ctx->h_cluster;
  STOCS_CUDA(ctx, cudaMemcpyAsync(&h->n, s.n, 4, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(h->kept, s.kept, (size_t)(p->maximum_pose_count + 1) * 8, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  *n_out = h->n;
  memcpy(index_out, h->kept, (size_t)h->n * 8);
  return STOCS_OK;
}
