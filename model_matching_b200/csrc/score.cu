// score.cu -- LCP scoring of rigid-transform hypotheses (the dominant kernel).
//
// Replaces stocs_estimator::compute_alignment_score_for_rigid_transform (reference
// src/stocs.cpp:1006-1041) and the kd-tree query it calls
// (include/super4pcs/accelerators/kdtree.h:394-459).
//
// One warp per hypothesis, persistent CTAs, dynamic work counter.  Model points live in shared
// memory as float4.
//   Phase A (per block of 256 model points; the top-K instantiation: over the whole model), two loops:
//     1. the test every point takes: fused affine map "transform o world->grid" (9 FMAs), floor,
//        block coordinates clamped to the always-empty border block (no bounds test, no branch),
//        one bit of a multi-resolution occupancy bitmap held in shared memory; survivors (~35 %)
//        are compacted, in model-point order, into a per-warp byte list (top-K: a survivor mask);
//     2. survivors only, 32 at a time: one bit of the per-brick bitmap, then -- occupied bricks
//        only -- ONE 16-byte brick record of the eps-dilated voxel grid (64-bit occupancy mask +
//        rank base); lanes whose cell is occupied are compacted (ballot + popc rank) into a
//        per-warp shared-memory queue that runs ACROSS rounds, in model-point order.
//   Phase B (queue more than half full, or end of the model), 32 queued queries at a time, one
//     per "owner" lane: (1) owners fetch their candidate-list offsets and compute the exact
//     transformed point; (2) the 32 candidate lists are swept as ONE flat list, 32 consecutive
//     float4 records per trip (coalesced, no padding to the longest list); owners are found with a
//     redux.or + popc, their points arrive by shuffle, hits race with shared-memory atomicMin on the
//     bit pattern of d^2 and then on the scene index; an exact d^2 tie falls through to a walk of
//     the reference kd-tree so that it is broken the way kdtree.h:416-428 breaks it; (3) owners
//     fetch the matched scene point's normal + class probability, apply the 30-degree test, and
//     the class probabilities are accumulated in lane order == model-point order, which makes the
//     LCP bit-identical to the reference's sequential fp32 sum.
// All memory-dependent steps are batched 32 wide, so the latency chain
// brick -> offsets -> candidates -> attributes is paid once per drain, not once per model point.
// The top-K instantiation (kPrune) also skips every hypothesis whose LCP provably stays below a
// value K other hypotheses of the launch reach: see prune_reject / prune_publish.
#include <cstring>

#include "stocs_ctx.h"

using namespace stocsm;

namespace {

constexpr int kWarps = 32;      // warps per CTA
constexpr int kMinBlocks = 2;   // CTAs per SM: 64 warps, which caps registers at 32
// queued queries per warp: a larger queue means fewer, fuller drains (S1: 64 -> 2.15 ms, 96 -> 2.09 ms,
// 128 -> 2.09 ms; shared memory per CTA grows by 8 KB per 32 entries)
constexpr int kQueue = 96;

struct ScoreArgs {
  const uint4* __restrict__ bricks;
  const uint32_t* __restrict__ coarse;   // 1 bit per block of 2^coarse_shift cells per axis: any occupied cell inside
  const uint32_t* __restrict__ brick_occ;  // 1 bit per brick: any occupied cell inside
  int coarse_words;                      // words of `coarse` (always staged in shared memory, <= 16 KB)
  int coarse_shift, coarse_nx, coarse_ny, coarse_nz;  // real blocks per axis; index n* is the empty border block
  int coarse_sx, coarse_sy;                           // row / slab strides of the map = blocks + 1
  const uint32_t* __restrict__ starts;
  const float4* __restrict__ cand;
  const float4* __restrict__ sattr;
  const float* __restrict__ model;   // 8*Mpad floats: float4 positions, then float4 normals
  const KdNodeDev* __restrict__ kd_nodes;
  const float4* __restrict__ kd_pts;
  const float* __restrict__ T;
  float* __restrict__ lcp;
  int* __restrict__ inl;
  unsigned long long* work_counter;
  unsigned long long* tie_counter;
  unsigned long long* cnt;   // counting variant only (stocs_b200_score_counters): see ScoreCounter
  const int* __restrict__ order;   // claim number -> hypothesis (heavy-first schedule, see probe_order_kernel) or NULL
  // top-K pruning (kPrune only, see prune_publish): theta bucket + histogram of this launch, the
  // context's two rejection counters, and the scene's bound constants
  unsigned* prune;                 // [0] theta bucket, [kBucketBase..] per-bucket counts; zeroed with the work counter
  unsigned long long* rejected;    // [0] after loop 1, [1] before a drain, [2] after loop 1b (accumulated over the context's lifetime)
  float w_max;                     // largest class weight of the scene
  float bound_scale;               // 1 + (M+2) 2^-23 (exact in fp32)
  unsigned key_lo;                 // bucket b >= 1 holds LCPs whose bit pattern >> 19 equals key_lo + b
  int K;
  long long H;
  const long long* __restrict__ H_dev;   // optional: the count lives on the device (H is then an upper bound)
  GridDesc g;
  int M, Mpad;
  float sq_eps, dot_thr;
  float to_block, to_cell;   // 2^-coarse_shift and 2^coarse_shift (exact scalings, see loop 1)
};

// kdtree.h:394-459 on the device (tie path only).
__device__ __noinline__ int kd_query_dev(const KdNodeDev* __restrict__ nodes, const float4* __restrict__ pts,
                                         float qx, float qy, float qz, float sqdist) {
  uint32_t st_node[64];
  float st_sq[64];
  int cl_id = -1;
  float cl_dist = sqdist;
  st_node[0] = 0; st_sq[0] = 0.f;
  unsigned count = 1;
  while (count) {
    uint32_t nid = st_node[count - 1];
    float sq = st_sq[count - 1];
    KdNodeDev nd = nodes[nid];
    if (sq < cl_dist) {
      if (nd.leaf) {
        --count;
        uint32_t end = nd.first_or_start + nd.dim_or_size;
        for (uint32_t i = nd.first_or_start; i < end; ++i) {
          float4 p = pts[i];
          float dx = qx - p.x, dy = qy - p.y, dz = qz - p.z;
          float d = dx * dx + (dy * dy + dz * dz);
          if (d <= cl_dist) { cl_dist = d; cl_id = __float_as_int(p.w); }
        }
      } else {
        float qd = nd.dim_or_size == 0 ? qx : (nd.dim_or_size == 1 ? qy : qz);
        float new_off = qd - nd.split;
        if (new_off < 0.f) {
          st_node[count] = nd.first_or_start;
          st_node[count - 1] = nd.first_or_start + 1;
        } else {
          st_node[count] = nd.first_or_start + 1;
          st_node[count - 1] = nd.first_or_start;
        }
        st_sq[count] = sq;
        st_sq[count - 1] = new_off * new_off;
        ++count;
      }
    } else {
      --count;
    }
  }
  return cl_id;
}

// Streaming 16-byte load that does not allocate in L1 (candidate and attribute records are read
// once per query; keeping them out of L1 leaves it to the brick table and the spill slots).
__device__ __forceinline__ float4 ld_stream(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}

// L2 policies.  With 0.5-eps cells the launch moves 12 GB through DRAM at ~4.4 TB/s and waits on
// memory (long scoreboard is the top stall), so L2 residency matters: brick records (70 MB at S1,
// re-used by every hypothesis) are loaded evict_last, candidate records (1.4 GB, touched once per
// query) evict_first: 2.58 -> 2.50 ms; the one-bit-per-brick filter in front of the brick record:
// 2.50 -> 2.48 ms.  (sm_100a accepts .L2::evict_* directly only on 256-bit loads, hence
// createpolicy + .L2::cache_hint.)
// the policy words are pure values (plain asm, so the compiler may hoist or rematerialise them)
__device__ __forceinline__ unsigned long long l2_policy_evict_last() {
  unsigned long long p;
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
  unsigned long long p;
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint4 ld_brick_keep(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(l2_policy_evict_last()));
  return v;
}
__device__ __forceinline__ float4 ld_cand_first(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(l2_policy_evict_first()));
  return v;
}

// %laneid / %lanemask_* as plain (non-volatile) asm: one instruction when the compiler has to
// rematerialise them inside the loops (registers are capped at 32 for 64 warps/SM)
__device__ __forceinline__ unsigned lane_id() { unsigned r; asm("mov.u32 %0, %%laneid;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned lanemask_lt() { unsigned r; asm("mov.u32 %0, %%lanemask_lt;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned lanemask_le() { unsigned r; asm("mov.u32 %0, %%lanemask_le;" : "=r"(r)); return r; }

struct WarpQueue {   // one per warp, shared memory (single base register, constant offsets)
  // exact transform and the same map into grid-block coordinates (FMA-evaluated, phase A only), as
  // three rows {m_r0, m_r1, m_r2, t_r}: a row is ONE 16-byte broadcast load (12 scalar loads per use
  // were a third of the kernel's shared-memory load wavefronts)
  float4 T[3];
  float4 G[3];
  uint32_t a0[kQueue];   // occupied-cell rank of the queued query
  uint32_t pi[kQueue];   // model point index of the queued query
  uint32_t best_d[32];   // drain: min over hits of the d^2 bit pattern (native 32-bit shared atomicMin)
  uint32_t best_i[32];   //        scene index of a candidate that attains it
  union {
    uint8_t plist[256];  // phase A: survivors of the coarse test within the current 256-point block
    struct {
      uint32_t wincl[32];  // loops 1b and 2: inclusive prefix of the survivor counts of a window of 32 mask words
      unsigned rej_brick;  // hypotheses this warp rejected after loop 1b
    } pr;                  // kPrune only
  };
  float thr_M;           // kPrune: theta * M rounded down (0: nothing to reject against)
  int later;             // kPrune: survivors in the windows after the current one
  unsigned rej[2];       // kPrune: hypotheses this warp rejected after loop 1 / before a drain
};
// (after the WarpQueues, kPrune: one survivor mask of Mpad/32 words per warp, bit = coarse-test survivor)

struct Acc { float acc; int inl; unsigned ties; };

// Model positions in shared memory as three float arrays x[Mpad] y[Mpad] z[Mpad]: a warp load is three
// LDS.32 = 3 wavefronts of the L1 data pipe -- the kernel's binding resource -- where a float4 record
// (LDS.128) takes 4, and a gather of 32 arbitrary points conflicts less (S1 2.074 -> 2.058 ms,
// S1-fit 3.582 -> 3.481 ms).
struct ModelPts {
  const float* x; int Mpad;
  __device__ __forceinline__ float4 operator[](int i) const { return make_float4(x[i], x[Mpad + i], x[2 * Mpad + i], 0.f); }
};
constexpr int kModelFloats = 3;   // floats of shared memory per (padded) model point

// Work counters of the counting variant (template parameter kCount; the timed kernel carries none
// of this).  One global atomic per warp-level event, issued by lane 0.
enum ScoreCounter { SC_SURVIVORS = 0, SC_BRICK_RECORDS, SC_QUEUED, SC_CANDIDATES, SC_HITS, SC_INLIERS, SC_DRAINS, SC_N };
static_assert(SC_N <= sizeof(DevScratch::score_counts) / 8, "DevScratch::score_counts holds every ScoreCounter");
template <bool kCount>
__device__ __forceinline__ void count(const ScoreArgs& a, int lane, int slot, unsigned v) {
  if (kCount) { if (lane == 0 && v) atomicAdd(a.cnt + slot, (unsigned long long)v); }
}

// Phase B, steps (1)-(3) of the file comment.  The queued queries are processed 32 at a time, one
// per lane ("owner" lane e holds query e: exact transformed point, candidate offset, candidate count).
// Step 1 computes the EXACT transformed point (mat * p.homogeneous()).head<3>() in the reference's
// evaluation order (stocs_math.h xform_point): phase A only located the cell.
template <bool kCount>
__device__ __forceinline__ void drain_queue(const ScoreArgs& a, WarpQueue& q, int qn, int lane,
                                            const ModelPts mp4, const float4* __restrict__ mn4, Acc& r) {
  __syncwarp();
  const float sq_eps = a.sq_eps;
  const unsigned le_mask = lanemask_le();
  for (int half = 0; half < qn; half += 32) {
    const int e = half + lane;
    const bool has = e < qn;
    // 1.
    uint32_t s = 0, cnt = 0, mi = 0;
    float qx = 0.f, qy = 0.f, qz = 0.f;
    if (has) {
      const uint32_t k = q.a0[e];
      s = __ldg(a.starts + k);
      cnt = __ldg(a.starts + k + 1) - s;
      mi = q.pi[e];
      const float4 mp = mp4[mi];
      const float4 t0 = q.T[0], t1 = q.T[1], t2 = q.T[2];
      qx = ((t0.x * mp.x + t0.y * mp.y) + t0.z * mp.z) + t0.w;
      qy = ((t1.x * mp.x + t1.y * mp.y) + t1.z * mp.z) + t1.w;
      qz = ((t2.x * mp.x + t2.y * mp.y) + t2.z * mp.z) + t2.w;
    }
    q.best_d[lane] = 0xffffffffu;
    uint32_t pre = cnt;         // inclusive scan of the counts -> exclusive prefix
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t up = __shfl_up_sync(0xffffffffu, pre, o);
      if (lane >= o) pre += up;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, pre, 31);
    pre -= cnt;
    count<kCount>(a, lane, SC_CANDIDATES, total);
    count<kCount>(a, lane, SC_DRAINS, 1u);
    __syncwarp();
    // 2.
    unsigned flag = 0;          // queries this lane wants answered by the kd-tree (exact d^2 ties)
    for (uint32_t t0 = 0; t0 < total; t0 += 32) {
      const uint32_t f = t0 + lane;
      const int rel = (int)pre - (int)t0;
      const unsigned starts_here = __reduce_or_sync(0xffffffffu, (cnt > 0 && rel >= 0 && rel < 32) ? (1u << rel) : 0u);
      const int before = __popc(__ballot_sync(0xffffffffu, cnt > 0 && rel < 0));
      // owner = the last query whose list starts at or before f.  Lists are non-empty (every queued
      // cell is occupied), so ranks among non-empty lists == lane numbers among `has` lanes.
      const int own = before - 1 + __popc(starts_here & le_mask);
      const int src = own < 0 ? 0 : own;
      const float ox = __shfl_sync(0xffffffffu, qx, src), oy = __shfl_sync(0xffffffffu, qy, src),
                  oz = __shfl_sync(0xffffffffu, qz, src);
      const uint32_t os = __shfl_sync(0xffffffffu, s, src), op = __shfl_sync(0xffffffffu, pre, src);
      bool hit = false;
      uint32_t hb = 0, hi = 0;
      if (f < total) {
        const float4 c = ld_cand_first(a.cand + (uint32_t)(os + (f - op)));
        const float dx = ox - c.x, dy = oy - c.y, dz = oz - c.z;
        const float d = dx * dx + (dy * dy + dz * dz);
        // (d^2 >= 0, so its bit pattern orders like the value.)  The minimum is taken with the
        // native 32-bit shared atomic; a candidate that meets its own d^2 already stored is an exact
        // tie (flag); after the trip's atomics, whoever equals the minimum records its index.  (A
        // 64-bit atomicMin on (d^2, index) compiles to a CAS loop: S1 2.28 -> 2.15 ms, S1-fit
        // 4.06 -> 3.76 ms with the 32-bit one.)
        hit = d <= sq_eps;
        hb = __float_as_uint(d); hi = __float_as_uint(c.w);
        if (hit && atomicMin(&q.best_d[src], hb) == hb) flag |= 1u << src;
      }
      __syncwarp();
      if (hit && q.best_d[src] == hb) q.best_i[src] = hi;
      __syncwarp();
    }
    __syncwarp();
    flag = __reduce_or_sync(0xffffffffu, flag);
    // 3.
    bool match = false;
    float w = 0.f;
    const bool found = q.best_d[lane] != 0xffffffffu;
    if (has && found) {
      int res = (int)q.best_i[lane];
      if ((flag >> lane) & 1u) {
        res = kd_query_dev(a.kd_nodes, a.kd_pts, qx, qy, qz, sq_eps);
        r.ties++;
      }
      if (res >= 0) {
        const float4 sa = ld_stream(a.sattr + res);
        const float4 mn = __ldg(mn4 + mi);
        // mat.block<3,3>(0,0) * n  -- see stocs_math.h xform_dir
        const float4 t0 = q.T[0], t1 = q.T[1], t2 = q.T[2];
        const float rx = t0.x * mn.x + (t0.y * mn.y + t0.z * mn.z);
        const float ry = t1.x * mn.x + (t1.y * mn.y + t1.z * mn.z);
        const float rz = t2.x * mn.x + (t2.y * mn.y + t2.z * mn.z);
        const float dt = sa.x * rx + (sa.y * ry + sa.z * rz);
        // acos(dt)*180/pi < 30  <=>  dot_thr <= dt <= 1   (threshold found by bisection on the host)
        match = (dt >= a.dot_thr) && (dt <= 1.0f);
        w = sa.w;
      }
    }
    unsigned mm = __ballot_sync(0xffffffffu, match);
    if (kCount) count<kCount>(a, lane, SC_HITS, __popc(__ballot_sync(0xffffffffu, has && found)));
    count<kCount>(a, lane, SC_INLIERS, __popc(mm));
    r.inl += __popc(mm);
    while (mm) {  // ordered fp32 accumulation == the reference's sequential loop
      const int b = __ffs(mm) - 1;
      r.acc += __shfl_sync(0xffffffffu, w, b);
      mm &= mm - 1;
    }
    __syncwarp();
  }
}

// next unit of work (lane 0 only): a claim number from the global counter, mapped through the
// heavy-first order when there is one; any value >= H ends the warp
__device__ __forceinline__ int claim_hypothesis(const ScoreArgs& a) {
  const unsigned long long c = atomicAdd(a.work_counter, 1ull);
  // (the online pipeline keeps its transform count on the device: H is then only an upper bound)
  const unsigned long long lim = a.H_dev ? (unsigned long long)__ldg(a.H_dev) : (unsigned long long)a.H;
  if (c >= lim) return 0x7fffffff;
  return a.order ? __ldg(a.order + c) : (int)c;
}

// position of the (r+1)-th set bit of w (r < popc(w))
__device__ __forceinline__ unsigned nth_set_bit(unsigned w, unsigned r) {
  unsigned pos = 0;
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const unsigned c = __popc(w & ((1u << s) - 1u));
    if (r >= c) { r -= c; w >>= s; pos += s; }
  }
  return pos;
}

// ---- Top-K pruning (kPrune: the caller receives nothing but the K best records) ----------------
// Bound.  The LCP is fl(S/M), S the fp32 sequential sum of the weights of the matched model points.
// When `acc` has been summed and at most n further weights, each in [0, w_max], can follow, then
// S <= (acc + n w_max)(1 + u)^n and fl(S/M) <= (S/M)(1 + u), u = 2^-24; for n <= M <= 5120,
// (1 + u)^(M+1) < 1 + (M+2) 2^-23 = bound_scale.  B below is evaluated with upward rounding, theta*M
// with downward rounding, so  B < theta*M  =>  lcp < theta  STRICTLY.  theta is a value that at least
// K fully scored hypotheses of this launch reach, so the hypothesis's key is below the K-th key and it
// cannot enter the top K; a hypothesis that could tie theta is never rejected, so ties are still
// decided by index.  theta > 0 whenever anything is rejected, and topk_kernel ignores lcp == 0, so the
// 0 written for a rejected hypothesis never displaces a record.
__device__ __forceinline__ bool prune_reject(const ScoreArgs& a, float acc, int n, float thr_M) {
  const float B = __fmul_ru(__fmaf_ru((float)n, a.w_max, acc), a.bound_scale);
  return B < thr_M;
}

// theta.  Buckets of the LCP's bit pattern >> 19 (16 per octave), the top one just above w_max, 8
// octaves deep; anything lower is bucket 0, which is never counted.  Bucket b >= 1 holds only values
// >= its lower edge, an exact float, so "K hypotheses counted in buckets >= b" means "K hypotheses
// reach edge(b)".  prune[0] is the highest such b found so far: it only grows, every value it takes
// is valid, and a warp that reads a stale one only rejects less.  (A per-CTA threshold would not do:
// a CTA sees a few dozen strong hypotheses in the whole launch, its K-th arrives too late.)
constexpr int kBuckets = 128;
constexpr int kBucketBase = 32;   // prune[] index of bucket 0 (theta sits alone in the first 128 bytes)
__device__ __forceinline__ float theta_M(const ScoreArgs& a, unsigned tb) {
  return tb ? __fmul_rd(__uint_as_float((a.key_lo + tb) << 19), (float)a.M) : 0.f;
}
// the current theta bucket, read by lane 0 and broadcast: every lane takes the same branch on it even
// when another warp raises theta meanwhile
__device__ __forceinline__ unsigned theta_bucket(const ScoreArgs& a, int lane) {
  return __reduce_max_sync(0xffffffffu, lane == 0 ? __ldcg(a.prune) : 0u);
}
__device__ __forceinline__ unsigned lcp_bucket(const ScoreArgs& a, float v) {
  const unsigned k = __float_as_uint(v) >> 19;
  return k <= a.key_lo ? 0u : min(k - a.key_lo, (unsigned)kBuckets - 1u);
}
// a fully scored hypothesis in bucket b (>= 1, >= tb, the theta bucket this warp read) counts itself,
// then walks down from the top bucket, 32 buckets at a time, to the highest bucket that holds >= K
__device__ __forceinline__ void prune_publish(const ScoreArgs& a, unsigned b, unsigned tb, int lane) {
  unsigned* hist = a.prune + kBucketBase;
  if (lane == 0) atomicAdd(hist + b, 1u);
  __syncwarp();
  unsigned cum = 0;
  for (int top = kBuckets - 32; top >= 0 && (unsigned)(top + 31) > tb; top -= 32) {
    unsigned s = __ldcg(hist + top + lane);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {   // suffix sum: buckets >= top + lane
      const unsigned dn = __shfl_down_sync(0xffffffffu, s, o);
      if (lane + o < 32) s += dn;
    }
    s += cum;
    const unsigned ok = __ballot_sync(0xffffffffu, s >= (unsigned)a.K);
    if (ok) {
      const unsigned nb = (unsigned)top + 31u - __clz(ok);
      if (lane == 0 && nb > tb) atomicMax(a.prune, nb);
      return;
    }
    cum = __shfl_sync(0xffffffffu, s, 0);
  }
}

template <bool kCount, bool kPrune>
__global__ void __launch_bounds__(kWarps * 32, kMinBlocks) score_lcp_kernel(ScoreArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_model = reinterpret_cast<float*>(smem_raw);
  const int Mpad = a.Mpad;
  const int lane = (int)lane_id();
  // warp index through redux: the result lives in a UNIFORM register, and so does everything
  // derived from it (the warp's queue address), outside the 32-register budget -- as a plain
  // tid >> 5 the queue address was spilled and re-loaded at 18 sites (37 local loads per hypothesis)
  const int warp = (int)__reduce_max_sync(0xffffffffu, threadIdx.x >> 5);
  // dynamic shared memory: [model positions x[Mpad] y[Mpad] z[Mpad]][coarse bitmap][one WarpQueue per warp]
  for (int i = threadIdx.x; i < 4 * Mpad; i += blockDim.x) { const int c = i & 3; if (c < 3) s_model[c * Mpad + (i >> 2)] = a.model[i]; }
  uint32_t* s_coarse = reinterpret_cast<uint32_t*>(s_model + kModelFloats * Mpad);   // Mpad % 64 == 0: 16-byte aligned
  for (int i = threadIdx.x; i < a.coarse_words; i += blockDim.x) s_coarse[i] = a.coarse[i];
  WarpQueue* queues = reinterpret_cast<WarpQueue*>(s_coarse + ((a.coarse_words + 3) & ~3));
  WarpQueue& q = queues[warp];
  uint32_t* smask = reinterpret_cast<uint32_t*>(queues + kWarps) + warp * (Mpad >> 5);   // survivor mask
  if (kPrune && lane == 0) { q.rej[0] = 0u; q.rej[1] = 0u; q.pr.rej_brick = 0u; }
  __syncthreads();
  ModelPts mp4; mp4.x = s_model; mp4.Mpad = Mpad;                // positions as x[] y[] z[] (NaN beyond M)
  const float4* mn4 = reinterpret_cast<const float4*>(a.model) + Mpad;  // normals stay in global (hits only)

  const unsigned lt_mask = lanemask_lt();
  const int M = a.M;
  const int nw = (M + 31) >> 5;   // survivor-mask words (32 model points each)
  // shared-window address of the coarse bitmap, made warp-uniform through redux so that it lives in a
  // uniform register for the whole kernel
  const unsigned coarse_sa = __reduce_max_sync(0xffffffffu, (unsigned)__cvta_generic_to_shared(s_coarse));
  Acc r;
  r.ties = 0;

  // Work distribution: lane 0 claims the next hypothesis from the global counter when the warp has
  // finished one.  (Claiming ahead does not pay: the result cannot stay in a register across a
  // hypothesis at the 32-register cap, so the warp waits for the atomic either way -- 10 % of the
  // stall samples when it was a prefetch; claiming 4 or 8 at a time lengthens the tail by more
  // than it saves: 2.63 / 2.76 ms against 2.58 ms.)
  // (claimed index broadcast by redux for the same reason: h stays in a uniform register)
  int h = 0;
  if (lane == 0) h = claim_hypothesis(a);
  h = (int)__reduce_max_sync(0xffffffffu, (unsigned)h);
  while (h < a.H) {
    // lanes 0..11 fetch the 3x4 transform (column-major 4x4: element (r,c) at c*4+r) and publish
    // it, with its grid-coordinate version G = inv_cell * (T - origin), to the warp's shared slot
    if (lane < 12) {
      const int c = lane / 3, rr = lane - 3 * c;
      const float t = __ldg(a.T + 16 * (size_t)h + c * 4 + rr);
      const float o = (rr == 0) ? a.g.ox : (rr == 1 ? a.g.oy : a.g.oz);
      reinterpret_cast<float*>(q.T)[rr * 4 + c] = t;
      // G maps into BLOCK coordinates (cell coordinates * 2^-coarse_shift): loop 1 floors it straight
      // to the coarse-map index; loop 2 multiplies by 2^coarse_shift first.  Scaling by a power of two
      // commutes with every rounding of the FMA chain, so the cell found is bit-identical to mapping
      // with the unscaled G.
      reinterpret_cast<float*>(q.G)[rr * 4 + c] = ((c == 3) ? (t - o) * a.g.inv_cell : t * a.g.inv_cell) * a.to_block;
    }
    __syncwarp();
    // gK = element (row K % 3, column K / 3) of the grid map
    float4 gr0 = q.G[0], gr1 = q.G[1], gr2 = q.G[2];
    float g0 = gr0.x, g3 = gr0.y, g6 = gr0.z, g9 = gr0.w, g1 = gr1.x, g4 = gr1.y, g7 = gr1.z, g10 = gr1.w;
    float g2 = gr2.x, g5 = gr2.y, g8 = gr2.z, g11 = gr2.w;
    r.acc = 0.f;
    r.inl = 0;
    int qn = 0;
    // Phase A, two loops.  Loop 1 is the cheap test every point takes: fused affine map -> cell -> one
    // bit of the shared-memory coarse occupancy map.  Loop 2 visits only the survivors, 32 at a time in
    // model-point order: brick record, exact cell bit, enqueue.  (Explicit FMAs: the map only selects a
    // cell, the eps-dilation margin of the index absorbs its rounding; the exact point is recomputed
    // for queued queries.  Float->int floor saturates; NaN -- padding points, rejected fits -- gives
    // cell 0, whose queries find no candidate because every distance is NaN.)
    // loop 1 for model points p .. p+31: this lane's bit, and the warp's ballot in pm
    auto coarse_test = [&](int p, unsigned& pm) -> unsigned {
      const float4 mp = mp4[p + lane];
      const float fx = __fmaf_rn(g0, mp.x, __fmaf_rn(g3, mp.y, __fmaf_rn(g6, mp.z, g9)));
      const float fy = __fmaf_rn(g1, mp.x, __fmaf_rn(g4, mp.y, __fmaf_rn(g7, mp.z, g10)));
      const float fz = __fmaf_rn(g2, mp.x, __fmaf_rn(g5, mp.y, __fmaf_rn(g8, mp.z, g11)));
      const unsigned ix = (unsigned)__float2int_rd(fx), iy = (unsigned)__float2int_rd(fy), iz = (unsigned)__float2int_rd(fz);
      // block coordinates clamped to the always-empty border block (index = number of real
      // blocks): no bounds test, no branch; blocks left of the grid are huge as unsigned
      const unsigned cx = min(ix, (unsigned)a.coarse_nx), cy = min(iy, (unsigned)a.coarse_ny),
                     cz = min(iz, (unsigned)a.coarse_nz);
      const uint32_t cidx = (cz * (unsigned)a.coarse_sy + cy) * (unsigned)a.coarse_sx + cx;
      // The bitmap word is loaded through its shared-window address held in a uniform register, and
      // the ballot is written in PTX on ONE predicate: as plain C++ the compiler re-derived the
      // address (S2UR + UMOV + 2 ULEA) and a second predicate (ISETP) in every iteration -- 40 -> 35
      // SASS instructions per 32 points (profiles/r02_score_loop1_sass.txt).
      unsigned cw;
      asm("ld.shared.u32 %0, [%1];" : "=r"(cw) : "r"(coarse_sa + ((cidx >> 5) << 2)));
      const unsigned bitv = (cw >> (cidx & 31)) & 1u;
      asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\tvote.sync.ballot.b32 %0, p, 0xffffffff;\n\t}" : "=r"(pm) : "r"(bitv));
      return bitv;
    };
    // the brick of model point i's grid cell (and the cell's coordinates).
    // Loop 1b and loop 2 both take it from here: a survivor that loop 1b drops is one whose brick
    // loop 2 would have found empty.
    auto cell_of = [&](const float4 mp) -> uint3 {
      const float fx = __fmaf_rn(g0, mp.x, __fmaf_rn(g3, mp.y, __fmaf_rn(g6, mp.z, g9)));
      const float fy = __fmaf_rn(g1, mp.x, __fmaf_rn(g4, mp.y, __fmaf_rn(g7, mp.z, g10)));
      const float fz = __fmaf_rn(g2, mp.x, __fmaf_rn(g5, mp.y, __fmaf_rn(g8, mp.z, g11)));
      return make_uint3((unsigned)__float2int_rd(fx * a.to_cell), (unsigned)__float2int_rd(fy * a.to_cell),
                        (unsigned)__float2int_rd(fz * a.to_cell));
    };
    auto brick_index = [&](uint3 c) -> unsigned {
      return ((c.z >> 2) * (unsigned)a.g.nby + (c.y >> 2)) * (unsigned)a.g.nbx + (c.x >> 2);
    };
    auto brick_occupied = [&](unsigned bidx) -> bool { return (__ldg(a.brick_occ + (bidx >> 5)) >> (bidx & 31u)) & 1u; };
    // kPrune: loop 1b ran for this hypothesis, so every survivor left lies in an occupied brick
    bool refined = false;
    // loop 2 for the survivor model point i of this lane (valid lanes only); drains the queue when it
    // passes kQueue - 32.  kPrune: false = rejected before that drain (`unvisited` survivors of the
    // current window, and q.later of later windows, are still to come after this group)
    auto visit = [&](int i, bool valid, int unvisited) -> bool {
      const uint3 c = cell_of(mp4[i]);
      const unsigned ix = c.x, iy = c.y, iz = c.z;
      uint4 br = make_uint4(0u, 0u, 0u, 0u);
      const unsigned bidx = brick_index(c);
      // second-level filter: 1 bit per brick (L2-resident, 1/128 of the brick table) before the
      // 16 B brick record, which for an empty brick would be a wasted DRAM access
      const bool occupied = valid && ((kPrune && refined) || brick_occupied(bidx));
      if (occupied) br = ld_brick_keep(a.bricks + bidx);
      if (kCount) count<kCount>(a, lane, SC_BRICK_RECORDS, __popc(__ballot_sync(0xffffffffu, occupied)));
      const unsigned bit = ((iz & 3u) << 4) | ((iy & 3u) << 2) | (ix & 3u);
      const unsigned half = (bit & 32u) ? br.y : br.x;      // 64-bit occupancy mask as two words
      const bool has = (half >> (bit & 31u)) & 1u;
      const unsigned hm = __ballot_sync(0xffffffffu, has);
      if (hm) {
        if (has) {
          const int slot = qn + __popc(hm & lt_mask);
          const unsigned below = __popc(half & ((1u << (bit & 31u)) - 1u)) + ((bit & 32u) ? __popc(br.x) : 0u);
          q.a0[slot] = br.z + below;
          q.pi[slot] = (uint32_t)i;
        }
        qn += __popc(hm);
        count<kCount>(a, lane, SC_QUEUED, __popc(hm));
      }
      if (qn > kQueue - 32) {
        // at most the queued queries and the survivors not yet visited can still add a weight
        if (kPrune && prune_reject(a, r.acc, qn + q.later + max(unvisited, 0), q.thr_M)) return false;
        // drain whole groups of 32 only; the (in-order) remainder stays at the front of the queue,
        // so a hypothesis pays for a partly filled group once, at its end (S1 2.098 -> 2.082 ms,
        // S1-fit 3.660 -> 3.611 ms)
        const int full = qn & ~31;
        drain_queue<kCount>(a, q, full, lane, mp4, mn4, r);
        const int rem = qn - full;
        uint32_t ca = 0, cp = 0;
        if (lane < rem) { ca = q.a0[full + lane]; cp = q.pi[full + lane]; }
        __syncwarp();
        if (lane < rem) { q.a0[lane] = ca; q.pi[lane] = cp; }
        __syncwarp();
        qn = rem;
        // the map is re-read after a drain so that it is not live (in registers) across it
        gr0 = q.G[0]; gr1 = q.G[1]; gr2 = q.G[2];
        g0 = gr0.x; g3 = gr0.y; g6 = gr0.z; g9 = gr0.w; g1 = gr1.x; g4 = gr1.y; g7 = gr1.z; g10 = gr1.w;
        g2 = gr2.x; g5 = gr2.y; g8 = gr2.z; g11 = gr2.w;
      }
      return true;
    };
    if (!kPrune) {
      // per block of 256 model points: loop 1 compacts the survivors' indices, in model-point order,
      // into a per-warp byte list, loop 2 walks it
      for (int blk = 0; blk < M; blk += 256) {
        int nl = 0;
        const int rounds = min(8, (M - blk + 31) >> 5);
        for (int rr = 0; rr < rounds; ++rr) {
          unsigned pm;
          const bool pass = coarse_test(blk + rr * 32, pm) != 0u;
          if (pass) q.plist[nl + __popc(pm & lt_mask)] = (uint8_t)(rr * 32 + lane);
          nl += __popc(pm);
        }
        count<kCount>(a, lane, SC_SURVIVORS, (unsigned)nl);
        __syncwarp();
        for (int e0 = 0; e0 < nl; e0 += 32) {
          const bool valid = e0 + lane < nl;
          visit(blk + (valid ? (int)q.plist[e0 + lane] : 0), valid, 0);
        }
        __syncwarp();
      }
    } else {
      // kPrune: loop 1 runs over the WHOLE model first, so that the survivor count is known before the
      // first brick lookup; the ballot of every 32 points is one word of the warp's survivor mask
      for (int rr = 0; rr < nw; ++rr) {
        unsigned pm;
        coarse_test(rr * 32, pm);
        if (lane == 0) smask[rr] = pm;
      }
      __syncwarp();
      unsigned ns = 0;   // survivors of the whole model
      for (int j = 0; j < nw; j += 32) ns += j + lane < nw ? __popc(smask[j + lane]) : 0u;
      ns = __reduce_add_sync(0xffffffffu, ns);
      const float thr = theta_M(a, theta_bucket(a, lane));
      if (prune_reject(a, 0.f, (int)ns, thr)) {
        if (lane == 0) q.rej[0]++;
        goto rejected;
      }
      {
        // inclusive prefix of the survivor counts of mask words wb .. wb+31 into q.pr.wincl (this lane's
        // prefix is returned)
        auto window_prefix = [&](int wb) -> unsigned {
          unsigned s = wb + lane < nw ? __popc(smask[wb + lane]) : 0u;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const unsigned up = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += up;
          }
          q.pr.wincl[lane] = s;
          return s;
        };
        // model point of survivor e (clamped to wn - 1) of the window at wb: its word is the first whose
        // inclusive prefix exceeds e
        auto survivor = [&](int wb, int wn, int e) -> int {
          const unsigned k = (unsigned)min(e, wn - 1);
          unsigned wj = 0;
#pragma unroll
          for (int st = 16; st >= 1; st >>= 1)
            if (q.pr.wincl[wj + st - 1] <= k) wj += st;
          const unsigned word = smask[wb + wj];
          return (int)((wb + wj) * 32u + nth_set_bit(word, k - (q.pr.wincl[wj] - __popc(word))));
        };
        // Loop 1b: drop from the mask every survivor whose brick is empty (loop 2 would queue nothing for
        // it, so the queue, the drains and the LCP are unchanged), then bound again on what is left.  Only
        // for a hypothesis the refined count may reject: a pose with many survivors is one on scene
        // surface, whose bricks are occupied anyway.  The gate -- half the survivors would be rejected
        // -- only decides whether the bound is tried (B200, S1 kernel: 1.073 ms; gate at 1/3 1.090 ms,
        // 2/3 1.083 ms, 5/6 1.114 ms, always 1.107 ms, none 1.145 ms).
        if (prune_reject(a, 0.f, (int)(ns / 2u), thr)) {
          int kept = 0, left = (int)ns;   // survivors kept so far / not examined yet
          for (int wb = 0; wb < nw; wb += 32) {
            window_prefix(wb);
            q.a0[lane] = 0u;   // the window's refined mask words (the queue stays empty until loop 2)
            __syncwarp();
            const int wn = (int)q.pr.wincl[31];
            // two survivors per lane, both brick-bit loads in flight before either is used; a lane past
            // the end loads the last survivor's word again and keeps nothing
            for (int e0 = 0; e0 < wn; e0 += 64) {
              const int e = e0 + lane;
              const int i0 = survivor(wb, wn, e), i1 = survivor(wb, wn, e + 32);
              const unsigned b0 = brick_index(cell_of(mp4[i0])), b1 = brick_index(cell_of(mp4[i1]));
              const unsigned w0 = __ldg(a.brick_occ + (b0 >> 5)), w1 = __ldg(a.brick_occ + (b1 >> 5));
              const bool o0 = e < wn && ((w0 >> (b0 & 31u)) & 1u), o1 = e + 32 < wn && ((w1 >> (b1 & 31u)) & 1u);
              if (o0) atomicOr(&q.a0[(i0 >> 5) - wb], 1u << (i0 & 31));
              if (o1) atomicOr(&q.a0[(i1 >> 5) - wb], 1u << (i1 & 31));
              kept += __popc(__ballot_sync(0xffffffffu, o0)) + __popc(__ballot_sync(0xffffffffu, o1));
              left -= min(wn - e0, 64);
              if (prune_reject(a, 0.f, kept + left, thr)) {   // left == 0 at the end: the bound on the refined count
                if (lane == 0) q.pr.rej_brick++;
                goto rejected;
              }
            }
            __syncwarp();
            if (wb + lane < nw) smask[wb + lane] = q.a0[lane];
            __syncwarp();
          }
          ns = (unsigned)kept;
          refined = true;
        }
        if (lane == 0) { q.thr_M = thr; q.later = (int)ns; }
        __syncwarp();
        // loop 2 over windows of 32 mask words (1024 model points)
        for (int wb = 0; wb < nw; wb += 32) {
          const unsigned s = window_prefix(wb);
          if (lane == 31) q.later -= (int)s;   // survivors in later windows
          __syncwarp();
          const int wn = (int)q.pr.wincl[31];
          for (int e0 = 0; e0 < wn; e0 += 32) {
            const bool valid = e0 + lane < wn;
            const int i = survivor(wb, wn, e0 + lane);
            if (!visit(valid ? i : 0, valid, wn - e0 - 32)) {
              if (lane == 0) q.rej[1]++;
              goto rejected;
            }
          }
          __syncwarp();
        }
      }
    }
    if (qn > 0) {
      if (kPrune && prune_reject(a, r.acc, qn, q.thr_M)) {
        if (lane == 0) q.rej[1]++;
        goto rejected;
      }
      drain_queue<kCount>(a, q, qn, lane, mp4, mn4, r);
    }
    {
      const float v = r.acc / (float)M;
      if (lane == 0) {
        a.lcp[h] = v;
        if (a.inl) a.inl[h] = r.inl;
      }
      if (kPrune) {
        const unsigned b = lcp_bucket(a, v), tb = theta_bucket(a, lane);
        if (b != 0u && b >= tb) prune_publish(a, b, tb, lane);
      }
    }
    if (false) {
    rejected:   // (kPrune only) lcp 0: topk_kernel never selects it
      if (lane == 0) {
        a.lcp[h] = 0.f;
        if (a.inl) a.inl[h] = 0;
      }
    }
    h = 0;
    if (lane == 0) h = claim_hypothesis(a);
    h = (int)__reduce_max_sync(0xffffffffu, (unsigned)h);
    __syncwarp();
  }
  if (r.ties) atomicAdd(a.tie_counter, (unsigned long long)r.ties);
  if (kPrune && lane == 0) {
    if (q.rej[0]) atomicAdd(a.rejected, (unsigned long long)q.rej[0]);
    if (q.rej[1]) atomicAdd(a.rejected + 1, (unsigned long long)q.rej[1]);
    if (q.pr.rej_brick) atomicAdd(a.rejected + 2, (unsigned long long)q.pr.rej_brick);
  }
}

// Heavy-first schedule.  The cost of a hypothesis varies by an order of magnitude (a pose that lands
// the model on scene surface queues hundreds of queries, a pose in free space none), and with one
// warp per hypothesis the launch ends when the last HEAVY hypothesis claimed does: a straggler tail
// of ~0.09 ms, a quarter of the launch when 10^6 hypotheses are sharded over 8 GPUs.  This kernel
// estimates the cost of every hypothesis from 32 sample points of the model (coarse-map test only:
// 1/16 of loop 1, about 1 % of the scoring work) and writes a claim order with the predicted-heavy
// hypotheses first and the light ones last.  The order only changes WHO scores a hypothesis WHEN;
// every result is computed exactly as before.
__global__ void __launch_bounds__(256) probe_order_kernel(ScoreArgs a, int* __restrict__ order, unsigned* __restrict__ fill,
                                                          int heavy_threshold) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4* s_pts = reinterpret_cast<float4*>(smem_raw);                 // 32 sample points
  uint32_t* s_coarse = reinterpret_cast<uint32_t*>(s_pts + 32);
  if (threadIdx.x < 32) s_pts[threadIdx.x] = reinterpret_cast<const float4*>(a.model)[(int)(((long long)threadIdx.x * a.M) / 32)];
  for (int i = threadIdx.x; i < a.coarse_words; i += blockDim.x) s_coarse[i] = a.coarse[i];
  __syncthreads();
  const long long h = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = lane_id();
  bool heavy = false;
  if (h < a.H) {
    float g[12];
    const float* t = a.T + 16 * (size_t)h;
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int rr = 0; rr < 3; ++rr) {
        const float v = __ldg(t + c * 4 + rr);
        const float o = (rr == 0) ? a.g.ox : (rr == 1 ? a.g.oy : a.g.oz);
        g[rr * 4 + c] = ((c == 3) ? (v - o) * a.g.inv_cell : v * a.g.inv_cell) * a.to_block;
      }
    int cnt = 0;
#pragma unroll 4
    for (int s = 0; s < 32; ++s) {
      const float4 mp = s_pts[s];
      const float fx = __fmaf_rn(g[0], mp.x, __fmaf_rn(g[1], mp.y, __fmaf_rn(g[2], mp.z, g[3])));
      const float fy = __fmaf_rn(g[4], mp.x, __fmaf_rn(g[5], mp.y, __fmaf_rn(g[6], mp.z, g[7])));
      const float fz = __fmaf_rn(g[8], mp.x, __fmaf_rn(g[9], mp.y, __fmaf_rn(g[10], mp.z, g[11])));
      const unsigned cx = min((unsigned)__float2int_rd(fx), (unsigned)a.coarse_nx), cy = min((unsigned)__float2int_rd(fy), (unsigned)a.coarse_ny),
                     cz = min((unsigned)__float2int_rd(fz), (unsigned)a.coarse_nz);
      const uint32_t cidx = (cz * (unsigned)a.coarse_sy + cy) * (unsigned)a.coarse_sx + cx;
      cnt += (s_coarse[cidx >> 5] >> (cidx & 31)) & 1u;
    }
    heavy = cnt >= heavy_threshold;
  }
  // warp-aggregated append: heavy hypotheses fill the order from the front, light ones from the back
  const unsigned valid = __ballot_sync(0xffffffffu, h < a.H);
  const unsigned hm = __ballot_sync(0xffffffffu, heavy);
  const unsigned lm = valid & ~hm;
  unsigned base_h = 0, base_l = 0;
  if (lane == 0) {
    if (hm) base_h = atomicAdd(&fill[0], (unsigned)__popc(hm));
    if (lm) base_l = atomicAdd(&fill[1], (unsigned)__popc(lm));
  }
  base_h = __shfl_sync(0xffffffffu, base_h, 0);
  base_l = __shfl_sync(0xffffffffu, base_l, 0);
  if (h < a.H) {
    const unsigned below = lanemask_lt();
    if (heavy) order[base_h + __popc(hm & below)] = (int)h;
    else order[(unsigned)a.H - 1u - (base_l + __popc(lm & below))] = (int)h;
  }
}

__global__ void fmad_selftest_kernel(float a, float b, float c, float* out) { out[0] = a * b + c; }

}  // namespace

bool stocs_fmad_selftest(stocs_b200_ctx* ctx) {
  // a*b = 1 + 2^-11 + 2^-24 rounds to 1 + 2^-11 (ties-to-even); unfused a*b+c == 0, fused == 2^-24.
  float* d = &ctx->scratch()->fmad_selftest;
  const float a = 1.0f + 1.0f / 4096.0f, c = -(1.0f + 1.0f / 2048.0f);
  fmad_selftest_kernel<<<1, 1, 0, ctx->stream>>>(a, a, c, d);
  float hres = 1.f;
  if (cudaMemcpyAsync(&hres, d, 4, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) return false;
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return false;
  return hres == 0.0f;
}

int stocs_launch_score(stocs_b200_ctx* ctx, const float* d_T, int64_t H, float* d_lcp, int32_t* d_inl,
                       cudaStream_t st, const ScoreRequest& rq) {
  if (H <= 0) return STOCS_OK;
  if (H >= (1ll << 31)) STOCS_FAIL(ctx, STOCS_E_ARG, "score: at most 2^31-1 hypotheses per call");
  // the pruned instantiation exists for one launch shape: slot 0, count on the host, no counting
  if (rq.top_K > 0 && (rq.counters || rq.d_H || rq.slot != 0))
    STOCS_FAIL(ctx, STOCS_E_ARG, "score: a top-K launch takes no counters, device count or slot");
  const int slot = rq.slot;
  unsigned long long* const d_counters = rq.counters;
  const long long* const d_H = rq.d_H;
  // the kd-tree of a freshly uploaded scene may still be under construction on a host thread: collect
  // it and queue its upload in front of this launch (no-op on every later launch)
  if (ctx->kd_pending) { const int rc = stocs_kd_finish(ctx, st); if (rc) return rc; }
  ScoreArgs a;
  a.bricks = ctx->d_bricks.as<uint4>();
  a.coarse = ctx->d_coarse.as<uint32_t>();
  a.brick_occ = ctx->d_brick_occ.as<uint32_t>();
  a.coarse_words = ctx->coarse_words;
  a.coarse_shift = ctx->coarse_shift; a.coarse_nx = ctx->coarse_nx; a.coarse_ny = ctx->coarse_ny; a.coarse_nz = ctx->coarse_nz;
  a.coarse_sx = ctx->coarse_nx + 1; a.coarse_sy = ctx->coarse_ny + 1;
  a.starts = ctx->d_cell_start.as<uint32_t>();
  a.cand = ctx->d_cand.as<float4>();
  a.sattr = ctx->d_sattr.as<float4>();
  a.model = ctx->d_model.as<float>();
  a.kd_nodes = ctx->d_kd_nodes.as<KdNodeDev>();
  a.kd_pts = ctx->d_kd_pts.as<float4>();
  a.T = d_T;
  a.lcp = d_lcp;
  a.inl = d_inl;
  // slot 0 is the default work counter; launches that may run concurrently (staged host-buffer chunks
  // on two streams) take distinct slots.  One tie counter accumulates over all launches.
  DevScratch* scr = ctx->scratch();
  unsigned long long* wctr = &scr->work[slot];
  a.work_counter = wctr;
  a.tie_counter = &scr->score_totals.ties;
  a.cnt = d_counters;
  a.order = nullptr;
  a.H = H;
  a.H_dev = d_H;
  a.g = ctx->grid;
  a.M = ctx->M;
  a.Mpad = ctx->Mpad;
  a.sq_eps = ctx->eps * ctx->eps;
  a.dot_thr = ctx->dot_thr;
  a.to_block = 1.0f / (float)(1u << ctx->coarse_shift);
  a.to_cell = (float)(1u << ctx->coarse_shift);
  // top-K pruning: only for a caller that receives nothing but the K best records (top_K = K), and
  // only on a scene whose class weights are all finite and >= 0 (the bound needs w_max)
  // (and with the lowest bucket edge a normal float, see lcp_bucket)
  unsigned wbits;
  memcpy(&wbits, &ctx->w_max, 4);
  const int key_lo = (int)(wbits >> 19) + 1 - (kBuckets - 1);
  const bool prune = rq.top_K > 0 && ctx->prune_ok && key_lo >= 16;
  a.prune = nullptr;
  a.rejected = scr->score_totals.rejected;
  a.w_max = ctx->w_max;
  a.bound_scale = 1.0f + (float)(ctx->M + 2) * 0x1p-23f;   // exact: M + 2 < 2^13
  a.key_lo = (unsigned)key_lo;
  a.K = rq.top_K;
  if (prune) {
    // [0, 8) work counter, [128, 132) theta bucket, [256, 768) bucket counts: one memset per launch
    DevBuf& b = ctx->pool[POOL_SCORE_PRUNE];
    STOCS_CUDA(ctx, b.ensure(256 + kBuckets * 4));
    wctr = b.as<unsigned long long>();
    a.work_counter = wctr;
    a.prune = (unsigned*)(b.as<char>() + 128);
  }
  size_t smem = (size_t)kModelFloats * ctx->Mpad * 4 + (size_t)((a.coarse_words + 3) & ~3) * 4 +
                (size_t)kWarps * (sizeof(WarpQueue) + (prune ? (size_t)(ctx->Mpad / 32) * 4 : 0));   // + survivor masks
  // static (per-warp queues) + dynamic (model, coarse bitmap) may exceed the 48 KB default
  // d_counters != NULL selects the counting variant (same code + one global atomic per warp event)
  void (*kernel)(ScoreArgs) = d_counters ? score_lcp_kernel<true, false>
                                         : (prune ? score_lcp_kernel<false, true> : score_lcp_kernel<false, false>);
  STOCS_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  STOCS_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kWarps * 32, smem));
  if (per_sm < 1) STOCS_FAIL(ctx, STOCS_E_ARG, "score: model too large for shared memory");
  long long want = ((d_H && rq.grid_hint > 0 && rq.grid_hint < H ? rq.grid_hint : H) + kWarps - 1) / kWarps;
  long long grid = (long long)ctx->num_sms * per_sm;
  if (grid > want) grid = want;
  STOCS_CUDA(ctx, cudaMemsetAsync(wctr, 0, prune ? 256 + kBuckets * 4 : 8, st));  // tie counter accumulates
  // Heavy-first schedule for MID-SIZE launches only.  Measured on B200 (S1 hypotheses, kernel + probe):
  // 125 000 hypotheses (the per-GPU share of the named config on 8 GPUs) 0.347 -> 0.312 ms; 10^6
  // hypotheses 2.100 -> 2.139 ms (the probe costs 64 us per 10^6, the tail it removes is ~0.09 ms
  // whatever the size), and on the all-fitted S1-fit list the heavy-first order itself slows the
  // kernel by 2 % (3.622 -> 3.692 ms).  Small launches (the online pipeline's ~1 000 hypotheses)
  // cannot spare one more launch.  STOCS_NO_LPT=1 switches it off, STOCS_LPT_MAX overrides the bound.
  const bool no_lpt = getenv("STOCS_NO_LPT") != nullptr;
  const long long lpt_max = getenv("STOCS_LPT_MAX") ? atoll(getenv("STOCS_LPT_MAX")) : 300000;
  // (not when the transforms are read in place from page-locked host memory: the probe would pull
  // every transform over PCIe a second time -- measured 1.7e9 -> 0.9e9 hypotheses/s end to end on 8 GPUs)
  if (!no_lpt && !d_counters && !d_H && H >= 32768 && H <= lpt_max && slot == 0 && !stocs_host_alias(d_T)) {
    DevBuf& b_order = ctx->pool[POOL_SCORE_ORDER];
    STOCS_CUDA(ctx, b_order.ensure((size_t)H * 4));
    unsigned* fill = scr->lpt_fill;
    STOCS_CUDA(ctx, cudaMemsetAsync(fill, 0, sizeof(scr->lpt_fill), st));
    const size_t psm = 32 * 16 + (size_t)((a.coarse_words + 3) & ~3) * 4;
    probe_order_kernel<<<(unsigned)((H + 255) / 256), 256, psm, st>>>(a, b_order.as<int>(), fill, 16);
    a.order = b_order.as<int>();
  }
  if (rq.time_it) {  // next pair of the ring (events are created on first use)
    const int k = (int)(ctx->ev_count % stocs_b200_ctx::kEvRing);
    for (int j = 0; j < 2; ++j)
      if (!ctx->ev_ring[2 * k + j]) STOCS_CUDA(ctx, cudaEventCreate(&ctx->ev_ring[2 * k + j]));
    ctx->ev0 = ctx->ev_ring[2 * k];
    ctx->ev1 = ctx->ev_ring[2 * k + 1];
    STOCS_CUDA(ctx, cudaEventRecord(ctx->ev0, st));
  }
  kernel<<<(unsigned)grid, kWarps * 32, smem, st>>>(a);
  if (rq.time_it) { STOCS_CUDA(ctx, cudaEventRecord(ctx->ev1, st)); ctx->ev_count++; }
  STOCS_CUDA(ctx, cudaGetLastError());
  ctx->counters[CTR_SCORE_LAUNCHES] += 1;
  ctx->timing_valid = rq.time_it;
  return STOCS_OK;
}
