// scene_index.cu -- scene centring and nearest-neighbour index construction on the device.
//
// Layout in HBM: cells are grouped in 4x4x4 bricks; the brick table holds {64-bit occupancy mask,
// rank of the brick's first occupied cell} (16 B per brick, ~1 MB for the 1M-point scene, the
// only structure every query touches), `starts` holds one offset per OCCUPIED cell, and the
// float4 candidate records follow in the same order.
//
// Replaces stocs_estimator::centroid_shift (reference src/stocs.cpp:943-964) and
// stocs_estimator::kdtree_initialize (src/stocs.cpp:966-980).  The NN index the scoring kernel
// reads is a dense voxel grid whose cells carry eps-DILATED candidate lists: cell C lists every
// scene point within eps (plus a rounding margin) of C's box, so an exact radius-eps query reads
// ONE cell descriptor and one contiguous run of float4 candidates.  The reference kd-tree
// (kdtree.h:355-370,522-641) is also built -- on the host, once per frame -- and uploaded; the
// scoring kernel walks it only when two candidates are at exactly the same squared distance, to
// reproduce the reference's traversal-order tie rule (kdtree.h:416-428).
#include <cub/device/device_scan.cuh>

#include <cstdio>
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <thread>

#include "stocs_ctx.h"

namespace {

// Sequential fp32 centroid in index order (src/stocs.cpp:945-956).  The sums are order
// dependent, so the chain is serial: 256 threads stage 2048-point chunks into shared memory with
// coalesced loads and lanes 0..2 of warp 0 run the three dependent add chains out of it.
__global__ void centroid_seq_kernel(const float* __restrict__ pos3, int n, float* __restrict__ out3) {
  constexpr int CH = 2048;
  __shared__ float buf[CH * 3];
  float acc = 0.f;
  for (int base = 0; base < n; base += CH) {
    int cnt = min(CH, n - base);
    for (int t = threadIdx.x; t < cnt * 3; t += blockDim.x) buf[t] = pos3[(size_t)base * 3 + t];
    __syncthreads();
    if (threadIdx.x < 3) {
      for (int i = 0; i < cnt; ++i) acc += buf[i * 3 + threadIdx.x];
    }
    __syncthreads();
  }
  if (threadIdx.x < 3) out3[threadIdx.x] = acc / (float)n;
}

__device__ __forceinline__ int f2ord(float f) {
  int i = __float_as_int(f);
  return i >= 0 ? i : i ^ 0x7fffffff;
}
__host__ __device__ __forceinline__ float ord2f(int i) {
  int b = i >= 0 ? i : i ^ 0x7fffffff;
  float f;
  memcpy(&f, &b, 4);
  return f;
}

// pos -= centroid (src/stocs.cpp:958-963); pack float4(x,y,z,bits(idx)); AABB via ordered ints.
__global__ void centre_pack_kernel(const float* __restrict__ pos3, int n, const float* __restrict__ c3,
                                   float4* __restrict__ out4, float* __restrict__ out3,
                                   int* __restrict__ aabb6) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  float cx = c3[0], cy = c3[1], cz = c3[2];
  int mn[3] = {INT_MAX, INT_MAX, INT_MAX}, mx[3] = {INT_MIN, INT_MIN, INT_MIN};
  if (i < n) {
    float x = pos3[3 * (size_t)i] - cx, y = pos3[3 * (size_t)i + 1] - cy, z = pos3[3 * (size_t)i + 2] - cz;
    out4[i] = make_float4(x, y, z, __int_as_float(i));
    if (out3) { out3[3 * (size_t)i] = x; out3[3 * (size_t)i + 1] = y; out3[3 * (size_t)i + 2] = z; }
    mn[0] = mx[0] = f2ord(x); mn[1] = mx[1] = f2ord(y); mn[2] = mx[2] = f2ord(z);
  }
  if (aabb6) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      int a = __reduce_min_sync(0xffffffffu, mn[k]);
      int b = __reduce_max_sync(0xffffffffu, mx[k]);
      if ((threadIdx.x & 31) == 0) { atomicMin(&aabb6[k], a); atomicMax(&aabb6[3 + k], b); }
    }
  }
}

__global__ void pack_attr_kernel(const float* __restrict__ nrm3, const float* __restrict__ cls, int n,
                                 float4* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = make_float4(nrm3[3 * (size_t)i], nrm3[3 * (size_t)i + 1], nrm3[3 * (size_t)i + 2], cls[i]);
}

// Cells are numbered brick-major: 4x4x4 bricks, 64 consecutive cell numbers per brick, so that a
// brick's occupancy fits one 64-bit mask and its candidate lists are contiguous.
__device__ __forceinline__ size_t cell_number(const GridDesc& g, int x, int y, int z) {
  const size_t brick = ((size_t)(z >> 2) * g.nby + (y >> 2)) * g.nbx + (x >> 2);
  return brick * 64 + (size_t)(((z & 3) << 4) | ((y & 3) << 2) | (x & 3));
}

struct CellRange { int x0, x1, y0, y1, z0, z1; };
__device__ __forceinline__ CellRange dilated_range(const GridDesc& g, float4 p, float r) {
  CellRange c;
  c.x0 = max(0, (int)floorf((p.x - r - g.ox) * g.inv_cell));
  c.x1 = min(g.nx - 1, (int)floorf((p.x + r - g.ox) * g.inv_cell));
  c.y0 = max(0, (int)floorf((p.y - r - g.oy) * g.inv_cell));
  c.y1 = min(g.ny - 1, (int)floorf((p.y + r - g.oy) * g.inv_cell));
  c.z0 = max(0, (int)floorf((p.z - r - g.oz) * g.inv_cell));
  c.z1 = min(g.nz - 1, (int)floorf((p.z + r - g.oz) * g.inv_cell));
  return c;
}

// squared distance from p to the box of cell (x,y,z): a point joins the cell's list only when it
// is within r of the box (Euclidean dilation; the per-axis ranges above are its bounding box)
__device__ __forceinline__ bool near_cell(const GridDesc& g, float4 p, float r2, int x, int y, int z) {
  const float cell = 1.0f / g.inv_cell;
  const float lx = g.ox + (float)x * cell, ly = g.oy + (float)y * cell, lz = g.oz + (float)z * cell;
  const float dx = fmaxf(fmaxf(lx - p.x, p.x - (lx + cell)), 0.f);
  const float dy = fmaxf(fmaxf(ly - p.y, p.y - (ly + cell)), 0.f);
  const float dz = fmaxf(fmaxf(lz - p.z, p.z - (lz + cell)), 0.f);
  return dx * dx + dy * dy + dz * dz <= r2;
}

// LPP lanes share one scene point and split the cells of its dilated range (LPP = 32 for frame-sized
// scenes: 13 419 threads walking ~150 cells each left the GPU idle for 90 us; LPP = 1 for large ones)
template <int LPP>
__global__ void grid_count_kernel(const float4* __restrict__ pts, int n, GridDesc g, float r,
                                  uint32_t* __restrict__ counts) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long i = t / LPP;
  const int sub = (int)(t % LPP);
  if (i >= n) return;
  const float4 p = pts[i];
  const CellRange c = dilated_range(g, p, r);
  const int nx = c.x1 - c.x0 + 1, ny = c.y1 - c.y0 + 1, nz = c.z1 - c.z0 + 1;
  if (nx <= 0 || ny <= 0 || nz <= 0) return;
  const int total = nx * ny * nz;
  for (int k = sub; k < total; k += LPP) {
    const int x = c.x0 + k % nx, y = c.y0 + (k / nx) % ny, z = c.z0 + k / (nx * ny);
    if (near_cell(g, p, r * r, x, y, z)) atomicAdd(&counts[cell_number(g, x, y, z)], 1u);
  }
}

// `remaining` holds the per-cell counts on entry: each record takes the next free slot of its cell from
// the back (no second zeroed cursor array; the order inside a cell's list is immaterial -- the scoring
// kernel takes the minimum distance and resolves exact ties through the kd-tree)
template <int LPP>
__global__ void grid_fill_kernel(const float4* __restrict__ pts, int n, GridDesc g, float r,
                                 const uint32_t* __restrict__ cell_start, uint32_t* __restrict__ remaining,
                                 float4* __restrict__ cand, uint32_t cap) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long i = t / LPP;
  const int sub = (int)(t % LPP);
  if (i >= n) return;
  const float4 p = pts[i];
  const CellRange c = dilated_range(g, p, r);
  const int nx = c.x1 - c.x0 + 1, ny = c.y1 - c.y0 + 1, nz = c.z1 - c.z0 + 1;
  if (nx <= 0 || ny <= 0 || nz <= 0) return;
  const int total = nx * ny * nz;
  for (int k = sub; k < total; k += LPP) {
    const int x = c.x0 + k % nx, y = c.y0 + (k / nx) % ny, z = c.z0 + k / (nx * ny);
    if (!near_cell(g, p, r * r, x, y, z)) continue;
    const size_t cell = cell_number(g, x, y, z);
    const uint32_t slot = cell_start[cell] + atomicSub(&remaining[cell], 1u) - 1u;
    if (slot < cap) cand[slot] = p;   // (the buffer is sized before the total is known; see stocs_build_scene_index)
  }
}

// per brick: occupancy mask and number of occupied cells.  One warp per 32 consecutive bricks, one
// brick per step: the 65 cell starts of a brick are two coalesced loads + one broadcast (a thread per
// brick read 65 words at a 256-byte stride: 89 us for the 21 M cells of the YCB frame).
__global__ void brick_mask_kernel(const uint32_t* __restrict__ cell_start, uint32_t nbricks,
                                  unsigned long long* __restrict__ masks, uint32_t* __restrict__ occ,
                                  uint32_t* __restrict__ brick_occ) {
  const int lane = threadIdx.x & 31;
  const uint32_t group = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // bricks 32*group .. 32*group + 31
  if ((size_t)group * 32 >= nbricks) return;
  uint32_t word = 0u;
  for (int t0 = 0; t0 < 32; t0 += 4) {   // 4 bricks per round: their 12 loads are issued together
    uint32_t v0[4], v1[4], v2[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t b = group * 32 + t0 + u;
      const uint32_t* cs = cell_start + (size_t)(b < nbricks ? b : nbricks - 1) * 64;
      v0[u] = cs[lane]; v1[u] = cs[32 + lane]; v2[u] = cs[64];
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t b = group * 32 + t0 + u;
      if (b >= nbricks) break;
      uint32_t n0 = __shfl_down_sync(0xffffffffu, v0[u], 1), n1 = __shfl_down_sync(0xffffffffu, v1[u], 1);
      const uint32_t first1 = __shfl_sync(0xffffffffu, v1[u], 0);
      if (lane == 31) { n0 = first1; n1 = v2[u]; }
      const unsigned lo = __ballot_sync(0xffffffffu, n0 != v0[u]), hi = __ballot_sync(0xffffffffu, n1 != v1[u]);
      const unsigned long long m = (unsigned long long)lo | ((unsigned long long)hi << 32);
      if (lane == 0) { masks[b] = m; occ[b] = (uint32_t)__popcll(m); }
      if (m) word |= 1u << (t0 + u);
    }
  }
  // 1 bit per brick: "has an occupied cell" (the scoring kernel's second-level filter)
  if (lane == 0) brick_occ[group] = word;
}

// brick table {mask lo, mask hi, index of the brick's first occupied cell, 0} + compact starts
__global__ void brick_table_kernel(const uint32_t* __restrict__ cell_start, const unsigned long long* __restrict__ masks,
                                   const uint32_t* __restrict__ occ_scan, uint32_t nbricks,
                                   const uint32_t* __restrict__ total_cand, uint32_t starts_cap,
                                   uint4* __restrict__ bricks, uint32_t* __restrict__ starts,
                                   uint32_t* __restrict__ coarse, GridDesc g, int cshift, int csx, int csy) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nbricks) return;
  const unsigned long long m = masks[b];
  if (m) {  // mark the coarse block (2^cshift cells per axis, cshift >= 2) this brick lies in
    const int bx = b % g.nbx, by = (b / g.nbx) % g.nby, bz = b / (g.nbx * g.nby);
    const int s = cshift - 2;
    const uint32_t cidx = (uint32_t)(((bz >> s) * csy + (by >> s)) * csx + (bx >> s));  // strides = blocks + 1
    atomicOr(&coarse[cidx >> 5], 1u << (cidx & 31));
  }
  const uint32_t base = occ_scan[b];
  bricks[b] = make_uint4((uint32_t)m, (uint32_t)(m >> 32), base, 0u);
  unsigned long long r = m;
  uint32_t k = base;
  while (r) {
    const int bit = __ffsll((long long)r) - 1;
    if (k < starts_cap) starts[k] = cell_start[(size_t)b * 64 + bit];
    ++k;
    r &= r - 1;
  }
  if (b == nbricks - 1 && occ_scan[nbricks] < starts_cap) starts[occ_scan[nbricks]] = *total_cand;
}

// Host construction of the reference kd-tree (explicit work stack instead of recursion; node
// numbering differs from the reference, tree shape and leaf point order do not).
struct KdBuild {
  std::vector<float> x, y, z;
  std::vector<int> idx;
  std::vector<KdNodeDev> nodes;
  const float* comp(unsigned d) const { return d == 0 ? x.data() : (d == 1 ? y.data() : z.data()); }

  // The reference's partition (kdtree.h:522-538) walks l up to the first element >= sv and r down to the
  // first element < sv, swaps them and repeats: it pairs the k-th misplaced element of the left part
  // with the k-th misplaced element, counted from the end, of the right part, where "left part" is the
  // first mid = #{c < sv} slots, and returns mid.  Written as count -> two branch-free compactions ->
  // swaps it produces the SAME permutation (checked against the loop form on 2*10^5 random arrays with
  // repeated values) at a third of the cost: the loop form mispredicts on every other element.
  std::vector<int> Lbuf, Rbuf;
  unsigned partition(int start, int end, unsigned dim, float sv) {
    const float* c = comp(dim);
    int mid = start;
    for (int i = start; i < end; ++i) mid += (c[i] < sv) ? 1 : 0;
    if ((int)Lbuf.size() < end - start) { Lbuf.resize((size_t)(end - start)); Rbuf.resize((size_t)(end - start)); }
    int nl = 0, nr = 0;
    int* L = Lbuf.data();
    int* R = Rbuf.data();
    for (int i = start; i < mid; ++i) { L[nl] = i; nl += (c[i] >= sv) ? 1 : 0; }
    for (int i = end - 1; i >= mid; --i) { R[nr] = i; nr += (c[i] < sv) ? 1 : 0; }
    for (int k = 0; k < nl; ++k) {   // nl == nr
      const int l = L[k], r = R[k];
      std::swap(x[l], x[r]); std::swap(y[l], y[r]); std::swap(z[l], z[r]);
      std::swap(idx[l], idx[r]);
    }
    return (unsigned)mid;
  }

  void build(const float* pos3, int n) {
    x.resize(n); y.resize(n); z.resize(n); idx.resize(n);
    for (int i = 0; i < n; ++i) { x[i] = pos3[3 * i]; y[i] = pos3[3 * i + 1]; z[i] = pos3[3 * i + 2]; idx[i] = i; }
    nodes.clear();
    nodes.push_back(KdNodeDev{0.f, 0u, 0u, 0u});
    struct Job { unsigned node, start, end, level; };
    std::vector<Job> todo;
    todo.push_back({0u, 0u, (unsigned)n, 1u});
    while (!todo.empty()) {
      Job j = todo.back();
      todo.pop_back();
      const float big = FLT_MAX / 2;
      float mn[3], mx[3];
      {  // bounding box of the node's points (scalars + selects: the compiler vectorises this form)
        const float* xs = x.data(); const float* ys = y.data(); const float* zs = z.data();
        float a0 = big, a1 = big, a2 = big, b0 = -big, b1 = -big, b2 = -big;
        for (unsigned i = j.start; i < j.end; ++i) {
          const float vx = xs[i], vy = ys[i], vz = zs[i];
          a0 = vx < a0 ? vx : a0; b0 = vx > b0 ? vx : b0;
          a1 = vy < a1 ? vy : a1; b1 = vy > b1 ? vy : b1;
          a2 = vz < a2 ? vz : a2; b2 = vz > b2 ? vz : b2;
        }
        mn[0] = a0; mn[1] = a1; mn[2] = a2; mx[0] = b0; mx[1] = b1; mx[2] = b2;
      }
      float hd[3] = {0.5f * (mx[0] - mn[0]), 0.5f * (mx[1] - mn[1]), 0.5f * (mx[2] - mn[2])};
      unsigned dim = 0;
      if (hd[1] > hd[dim]) dim = 1;
      if (hd[2] > hd[dim]) dim = 2;
      float sv = mn[dim] + ((mx[dim] - mn[dim]) / 2.0f);
      unsigned mid = partition((int)j.start, (int)j.end, dim, sv);
      unsigned first = (unsigned)nodes.size();
      nodes[j.node].split = sv;
      nodes[j.node].first_or_start = first;
      nodes[j.node].dim_or_size = dim;
      nodes[j.node].leaf = 0;
      nodes.push_back(KdNodeDev{0.f, 0u, 0u, 0u});
      nodes.push_back(KdNodeDev{0.f, 0u, 0u, 0u});
      unsigned lo[2] = {j.start, mid}, hi[2] = {mid, j.end};
      for (int c = 0; c < 2; ++c) {
        unsigned cnt = hi[c] - lo[c];
        if (cnt <= 64u || j.level >= 32u) {
          nodes[first + c].leaf = 1;
          nodes[first + c].first_or_start = lo[c];
          nodes[first + c].dim_or_size = cnt;
        } else {
          todo.push_back({first + (unsigned)c, lo[c], hi[c], j.level + 1});
        }
      }
    }
  }
};

}  // namespace

// Centre n points with the reference's sequential fp32 centroid; optional float4 / float3 device
// outputs, centroid and AABB (min xyz, max xyz of the centred points) returned to the host.
// h_pos3 (optional): the same points in host memory.  The centroid is an ORDER-DEPENDENT serial fp32
// sum (src/stocs.cpp:945-956), i.e. three dependent add chains of length n: one SM needs 5.5 ms for
// 2^20 points, a host core ~1.3 ms, and the host runs it while the H2D copy of the points is still in
// flight.  Without host data the single-CTA kernel does the same sum on the device.
// The reference kd-tree serves one purpose on the device: resolving EXACT distance ties in the scoring
// kernel.  Nothing before the first scoring launch needs it, so upload_scene starts its build (host
// work on the centred points, ~0.3 ms for a 13 000-point frame) on a host thread and returns once the
// grid index is complete; the first scoring launch -- in the online pipeline that is after base
// sampling, congruent sets and fits have been enqueued -- joins the thread and queues the upload in
// front of its kernel (stocs_kd_finish).  A new scene or the context's destruction joins it too.
struct KdPending {
  std::thread th;
  KdBuild kb;
  int S = 0;
  float4* pts = nullptr;                 // leaf-ordered points {x, y, z, bits(index)}: page-locked staging or `pageable`
  std::vector<float4> pageable;
  bool failed = false;
};

extern "C" int stocs_b200_host_kdtree_order(const float* pos3, int n, int32_t* leaf_order, int32_t* n_nodes) {
  if (!pos3 || n <= 0 || !leaf_order) return STOCS_E_ARG;
  KdBuild kb;
  kb.build(pos3, n);
  for (int i = 0; i < n; ++i) leaf_order[i] = kb.idx[i];
  if (n_nodes) *n_nodes = (int32_t)kb.nodes.size();
  return STOCS_OK;
}

int stocs_kd_finish(stocs_b200_ctx* ctx, cudaStream_t st, bool upload) {
  KdPending* kp = ctx->kd_pending;
  if (!kp) return STOCS_OK;
  if (kp->th.joinable()) kp->th.join();
  ctx->kd_pending = nullptr;
  struct Deleter { KdPending* p; ~Deleter() { delete p; } } del{kp};
  if (!upload) return STOCS_OK;
  if (kp->failed) STOCS_FAIL(ctx, STOCS_E_CUDA, "upload_scene: kd-tree construction failed (out of host memory)");
  const size_t node_bytes = kp->kb.nodes.size() * sizeof(KdNodeDev), pts_bytes = (size_t)kp->S * 16;
  ctx->kd_nodes = (int)kp->kb.nodes.size();
  STOCS_CUDA(ctx, ctx->d_kd_nodes.ensure(node_bytes));
  STOCS_CUDA(ctx, ctx->d_kd_pts.ensure(pts_bytes));
  // (pageable sources -- the node array always, the points of very large scenes -- have been consumed
  // when cudaMemcpyAsync returns; the page-locked staging buffer is guarded by kd_copy_done)
  STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->d_kd_nodes.p, kp->kb.nodes.data(), node_bytes, cudaMemcpyHostToDevice, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->d_kd_pts.p, kp->pts, pts_bytes, cudaMemcpyHostToDevice, st));
  if (!ctx->kd_copy_done) STOCS_CUDA(ctx, cudaEventCreateWithFlags(&ctx->kd_copy_done, cudaEventDisableTiming));
  STOCS_CUDA(ctx, cudaEventRecord(ctx->kd_copy_done, st));
  // scoring launches on the context's other streams (chunked host-buffer calls alternate between two) wait for it too
  for (cudaStream_t other : {ctx->stream, ctx->aux_stream})
    if (other && other != st) STOCS_CUDA(ctx, cudaStreamWaitEvent(other, ctx->kd_copy_done, 0));
  if (!kp->pageable.empty()) STOCS_CUDA(ctx, cudaStreamSynchronize(st));   // the pageable copy dies with kp
  return STOCS_OK;
}

// starts the build of the kd-tree over ctx->h_spos (S centred points) on a host thread
static int kd_start(stocs_b200_ctx* ctx, int S) {
  stocs_kd_finish(ctx, ctx->stream, false);
  const size_t pts_bytes = (size_t)S * 16;
  KdPending* kp = new (std::nothrow) KdPending();
  if (!kp) STOCS_FAIL(ctx, STOCS_E_CUDA, "upload_scene: out of host memory");
  kp->S = S;
  if (pts_bytes <= (size_t)(64u << 20)) {
    if (ctx->kd_copy_done) cudaEventSynchronize(ctx->kd_copy_done);   // the previous scene's upload has left the staging buffer
    if (ctx->h_kd_stage_bytes < pts_bytes) {
      if (ctx->h_kd_stage) cudaFreeHost(ctx->h_kd_stage);
      ctx->h_kd_stage = nullptr; ctx->h_kd_stage_bytes = 0;
      if (cudaHostAlloc(&ctx->h_kd_stage, pts_bytes * 2, cudaHostAllocDefault) != cudaSuccess) {
        delete kp;
        STOCS_FAIL(ctx, STOCS_E_CUDA, "upload_scene: page-locked allocation failed");
      }
      ctx->h_kd_stage_bytes = pts_bytes * 2;
    }
    kp->pts = (float4*)ctx->h_kd_stage;
  }
  const float* pos = ctx->h_spos.data();
  ctx->kd_pending = kp;
  kp->th = std::thread([kp, pos, S] {
    try {
      if (!kp->pts) { kp->pageable.resize((size_t)S); kp->pts = kp->pageable.data(); }
      kp->kb.build(pos, S);
      for (int i = 0; i < S; ++i) {
        float w;
        const int id = kp->kb.idx[i];
        memcpy(&w, &id, 4);
        kp->pts[i] = make_float4(kp->kb.x[i], kp->kb.y[i], kp->kb.z[i], w);
      }
    } catch (...) {
      kp->failed = true;
    }
  });
  return STOCS_OK;
}

int stocs_centre_points(stocs_b200_ctx* ctx, const float* d_pos3, int n, float4* d_out4,
                        float* d_out3, float* h_centroid3, float* h_aabb6, const float* h_pos3, float* h_centred3) {
  cudaStream_t st = ctx->stream;
  float* d_c = ctx->scratch()->centroid;
  int* d_aabb = ctx->scratch()->aabb;
  if (h_pos3) {
    float sx = 0.f, sy = 0.f, sz = 0.f;   // same order, same binary32 adds as the kernel (no contraction: no multiply)
    for (int i = 0; i < n; ++i) { sx += h_pos3[3 * (size_t)i]; sy += h_pos3[3 * (size_t)i + 1]; sz += h_pos3[3 * (size_t)i + 2]; }
    ctx->h_centroid_stage[0] = sx / (float)n; ctx->h_centroid_stage[1] = sy / (float)n; ctx->h_centroid_stage[2] = sz / (float)n;
    STOCS_CUDA(ctx, cudaMemcpyAsync(d_c, ctx->h_centroid_stage, 12, cudaMemcpyHostToDevice, st));
    if (h_centred3) {
      // The host has everything the callers wait for: centroid, centred copy (one binary32
      // subtraction per coordinate, the same operation as centre_pack_kernel) and bounding box.
      // The device centres its own copy concurrently; nothing is read back, no synchronisation.
      const float cx = ctx->h_centroid_stage[0], cy = ctx->h_centroid_stage[1], cz = ctx->h_centroid_stage[2];
      float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
      bool finite = true;
      for (int i = 0; i < n; ++i) {
        const float v[3] = {h_pos3[3 * (size_t)i] - cx, h_pos3[3 * (size_t)i + 1] - cy, h_pos3[3 * (size_t)i + 2] - cz};
        for (int k = 0; k < 3; ++k) {
          h_centred3[3 * (size_t)i + k] = v[k];
          if (v[k] < mn[k]) mn[k] = v[k];
          if (v[k] > mx[k]) mx[k] = v[k];
          finite = finite && std::isfinite(v[k]);
        }
      }
      if (!finite) mn[0] = NAN;   // callers test the box
      centre_pack_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_pos3, n, d_c, d_out4, d_out3, nullptr);
      STOCS_CUDA(ctx, cudaGetLastError());
      for (int k = 0; k < 3; ++k) h_centroid3[k] = ctx->h_centroid_stage[k];
      if (h_aabb6) for (int k = 0; k < 3; ++k) { h_aabb6[k] = mn[k]; h_aabb6[3 + k] = mx[k]; }
      return STOCS_OK;
    }
  } else {
    centroid_seq_kernel<<<1, 256, 0, st>>>(d_pos3, n, d_c);
  }
  int init[6] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN};
  STOCS_CUDA(ctx, cudaMemcpyAsync(d_aabb, init, sizeof(init), cudaMemcpyHostToDevice, st));
  centre_pack_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_pos3, n, d_c, d_out4, d_out3, d_aabb);
  STOCS_CUDA(ctx, cudaGetLastError());
  int haabb[6];
  STOCS_CUDA(ctx, cudaMemcpyAsync(h_centroid3, d_c, 12, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(haabb, d_aabb, 24, cudaMemcpyDeviceToHost, st));
  STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  if (h_aabb6)
    for (int k = 0; k < 6; ++k) h_aabb6[k] = ord2f(haabb[k]);
  return STOCS_OK;
}

int stocs_build_scene_index(stocs_b200_ctx* ctx) {
  // expects ctx->d_tmp = raw pos3 (S*3 floats)
  const int S = ctx->S_pending;   // committed to ctx->S by upload_scene once the index is complete
  cudaStream_t st = ctx->stream;
  StageTrace tr(st);
  STOCS_CUDA(ctx, ctx->d_spos4.ensure((size_t)S * 16));
  STOCS_CUDA(ctx, ctx->d_tmp2.ensure((size_t)S * 12));
  int nb = (S + 255) / 256;
  float aabb[6];
  ctx->h_spos.resize((size_t)S * 3);
  int rc = stocs_centre_points(ctx, ctx->d_tmp.as<float>(), S, ctx->d_spos4.as<float4>(),
                               ctx->h_pos_pending ? nullptr : ctx->d_tmp2.as<float>(), ctx->cs, aabb, ctx->h_pos_pending,
                               ctx->h_pos_pending ? ctx->h_spos.data() : nullptr);
  if (rc) return rc;
  if (!ctx->h_pos_pending) {   // device-only path: centred points and box come back from the kernels
    STOCS_CUDA(ctx, cudaMemcpyAsync(ctx->h_spos.data(), ctx->d_tmp2.p, (size_t)S * 12, cudaMemcpyDeviceToHost, st));
    STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  }
  tr.mark("centre + copy back");
  float mn[3] = {aabb[0], aabb[1], aabb[2]}, mx[3] = {aabb[3], aabb[4], aabb[5]};
  for (int k = 0; k < 3; ++k)
    if (!(mn[k] <= mx[k]) || !std::isfinite(mn[k]) || !std::isfinite(mx[k]))
      STOCS_FAIL(ctx, STOCS_E_ARG, "upload_scene: scene contains non-finite coordinates");

  // the reference kd-tree (exact-tie resolution in the scoring kernel): host work on the centred
  // points, started here on a host thread and collected by the first scoring launch
  rc = kd_start(ctx, S);
  if (rc) return rc;

  // grid geometry.  Cell edge in units of eps, measured on B200 with the S1 workload (10^6
  // hypotheses, all bit-identical): 2.0 -> 4.3 ms, 1.0 -> 2.93 ms, 0.6 -> 2.73 ms, 0.5 -> 2.64 ms,
  // 0.45 -> 2.62 ms, 0.405 -> 2.65 ms, 0.4 -> 3.46 ms (one more coarse-map level).  Smaller cells
  // mean shorter candidate lists (the list of a cell holds the points within eps of its box, a
  // volume of (c^3 + 6c^2 + 3*pi*c + 4.19) eps^3: 20.6 at c = 1, 10.5 at c = 0.5, against the
  // 4.19 of the query sphere itself) and a thinner occupied shell; a point is replicated into
  // that volume / c^3 lists and the tables grow with 1/c^3.  0.5 is the default: 84 candidate records per scene point
  // (1.4 GB at 2^20 points), 16 B of brick table per 64 cells.  The scale is raised until the
  // candidate records fit in 8 GB and the cells in kMaxCells.  STOCS_CELL_SCALE / STOCS_MAX_CELLS
  // override (tuning knobs).
  const double eps = ctx->eps;
  double kMaxCells = 512.0 * 1024 * 1024;
  if (const char* e = getenv("STOCS_MAX_CELLS")) { double v = atof(e); if (v >= 1e6 && v <= 4e9) kMaxCells = v; }
  double cell_scale = 0.5;
  if (const char* e = getenv("STOCS_CELL_SCALE")) { double v = atof(e); if (v >= 0.25 && v <= 16.0) cell_scale = v; }
  for (;;) {
    const double c = cell_scale;
    const double repl = (c * c * c + 6 * c * c + 3 * 3.14159265 * c + 4.19) / (c * c * c);
    if ((double)S * repl * 16.0 <= 8e9) break;
    cell_scale *= 1.25;
  }
  double cell = cell_scale * eps;
  double ext[3] = {(double)mx[0] - mn[0], (double)mx[1] - mn[1], (double)mx[2] - mn[2]};
  // apron: a query can lie up to eps outside the scene's bounding box and still have a neighbour,
  // so the grid extends floor(eps / cell) + 1 cells beyond the box on every side
  int apron = 2;
  for (;;) {
    apron = (int)floor(eps / cell) + 1;
    double n = (floor(ext[0] / cell) + 1 + 2 * apron) * (floor(ext[1] / cell) + 1 + 2 * apron) * (floor(ext[2] / cell) + 1 + 2 * apron);
    if (n <= kMaxCells) break;
    cell *= 1.25;
  }
  GridDesc g;
  g.ox = (float)(mn[0] - apron * cell); g.oy = (float)(mn[1] - apron * cell); g.oz = (float)(mn[2] - apron * cell);
  g.inv_cell = (float)(1.0 / cell);
  g.nx = (int)floor(ext[0] / cell) + 1 + 2 * apron; g.ny = (int)floor(ext[1] / cell) + 1 + 2 * apron;
  g.nz = (int)floor(ext[2] / cell) + 1 + 2 * apron;
  // Coarse occupancy map: blocks of 2^k cells per axis, k >= 2 (brick), smallest k whose bitmap
  // fits 16 KB.  The map is laid out with one extra, always-empty block per axis (index = number
  // of real blocks): the scoring kernel clamps block coordinates to it instead of testing grid
  // bounds (cells left of the grid are negative ints = huge unsigned values, so they clamp there
  // too).  The grid is padded to whole blocks so that "inside a real block" == "inside the grid".
  int cshift = 2, cnx = (g.nx + 3) >> 2, cny = (g.ny + 3) >> 2, cnz = (g.nz + 3) >> 2;
  size_t coarse_bits = 16 * 1024 * 8;
  if (const char* e = getenv("STOCS_COARSE_BITS")) { long v = atol(e); if (v >= 1024 && v <= 16 * 1024 * 8) coarse_bits = (size_t)v; }
  while ((size_t)(cnx + 1) * (cny + 1) * (cnz + 1) > coarse_bits) {
    ++cshift;
    cnx = (g.nx + (1 << cshift) - 1) >> cshift; cny = (g.ny + (1 << cshift) - 1) >> cshift; cnz = (g.nz + (1 << cshift) - 1) >> cshift;
  }
  g.nx = cnx << cshift; g.ny = cny << cshift; g.nz = cnz << cshift;
  g.nbx = (g.nx + 3) / 4; g.nby = (g.ny + 3) / 4; g.nbz = (g.nz + 3) / 4;
  g.nbricks = (uint32_t)((size_t)g.nbx * g.nby * g.nbz);
  g.ncells = g.nbricks * 64u;
  ctx->grid = g;
  // dilation radius: eps plus a margin that absorbs the rounding of both cell-index computations.
  // The scoring kernel locates cells through an FMA-evaluated affine map; its absolute error grows
  // with the magnitude of the cell coordinate (three chained binary32 FMAs: <= ~4 ulp of the largest
  // coordinate, i.e. 4 * n * 2^-24 cells on an axis of n cells): a few 1e-4 cells at S1 (830 cells),
  // but 0.02 cells on a long thin scene of 10^5 cells.  The margin is therefore
  // max(cell/256, 2 * that bound) + eps/256 -- cell/256 for every grid up to 32 768 cells per axis.
  const double nmax = (double)std::max(g.nx, std::max(g.ny, g.nz));
  const double margin_cells = std::max(1.0 / 256.0, 2.0 * 4.0 * nmax * 5.9604644775390625e-8);
  const float r = (float)(eps * (1.0 + 1.0 / 256.0) + cell * margin_cells);

  // Everything below is enqueued without a host round trip: the candidate buffer and the compact
  // cell-start array are sized BEFORE the device knows their lengths -- from the expected replication
  // (the volume formula above, +10 %), or from whatever an earlier scene left allocated if that is
  // larger -- writes beyond the capacity are dropped, and the two lengths come back with the single
  // synchronisation at the end; a scene that did not fit grows the buffers and runs the stage again.
  // (Round 1 synchronised four times here: candidate total, occupied-cell total, tables, kd-tree.)
  size_t nc1 = (size_t)g.ncells + 1;
  DevBuf& d_dense = ctx->pool[POOL_INDEX_DENSE];  // dense per-cell starts (scratch)
  STOCS_CUDA(ctx, d_dense.ensure(nc1 * 4));
  // per-cell counters: a buffer of their own that every build leaves ZEROED (the fill pass takes each
  // count back down to 0), so only its first use -- or a larger grid -- pays the memset (84 MB on the YCB frame)
  DevBuf& d_counts = ctx->pool[POOL_INDEX_COUNTS];
  if (d_counts.bytes < nc1 * 4) ctx->index_counts_clean = 0;
  STOCS_CUDA(ctx, d_counts.ensure(nc1 * 4));
  uint32_t* counts = d_counts.as<uint32_t>();
  uint32_t* dense_start = d_dense.as<uint32_t>();
  DevBuf &d_masks = ctx->pool[POOL_INDEX_MASKS], &d_occ = ctx->pool[POOL_INDEX_OCC], &d_occ_scan = ctx->pool[POOL_INDEX_OCC_SCAN];
  STOCS_CUDA(ctx, d_masks.ensure((size_t)g.nbricks * 8));
  STOCS_CUDA(ctx, d_occ.ensure((size_t)(g.nbricks + 1) * 4));
  STOCS_CUDA(ctx, d_occ_scan.ensure((size_t)(g.nbricks + 1) * 4));
  STOCS_CUDA(ctx, ctx->d_brick_occ.ensure(((size_t)g.nbricks + 31) / 32 * 4));
  STOCS_CUDA(ctx, ctx->d_bricks.ensure((size_t)g.nbricks * 16));
  ctx->coarse_shift = cshift; ctx->coarse_nx = cnx; ctx->coarse_ny = cny; ctx->coarse_nz = cnz;
  ctx->coarse_words = (int)(((size_t)(cnx + 1) * (cny + 1) * (cnz + 1) + 31) / 32);
  STOCS_CUDA(ctx, ctx->d_coarse.ensure((size_t)ctx->coarse_words * 4));
  size_t tmp_bytes = 0, tmp_bytes2 = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, counts, dense_start, (int)nc1, st);
  cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes2, d_occ.as<uint32_t>(), d_occ_scan.as<uint32_t>(), (int)(g.nbricks + 1), st);
  STOCS_CUDA(ctx, ctx->d_tmp2.ensure(tmp_bytes > tmp_bytes2 ? tmp_bytes : tmp_bytes2));
  const double cs_eff = cell / eps;
  const double repl = (cs_eff * cs_eff * cs_eff + 6 * cs_eff * cs_eff + 3 * 3.14159265 * cs_eff + 4.19) / (cs_eff * cs_eff * cs_eff);
  size_t cap = (size_t)((double)S * repl * 1.1) + 4096;
  if (cap < ctx->d_cand.bytes / 16) cap = ctx->d_cand.bytes / 16;
  if (const char* e = getenv("STOCS_CAND_CAP")) { const long long v = atoll(e); if (v >= 1) cap = (size_t)v; }   // tests: force the retry
  if (cap > 0xfffffff0u) cap = 0xfffffff0u;
  const unsigned bb = (g.nbricks + 127) / 128;
  uint32_t* h_counts = ctx->h_index_counts;   // page-locked: {candidate records, occupied cells}
  uint32_t total = 0, n_occ = 0;
  for (int attempt = 0;; ++attempt) {
    const size_t starts_cap = (cap < (size_t)g.ncells ? cap : (size_t)g.ncells) + 1;
    STOCS_CUDA(ctx, ctx->d_cand.ensure(cap * 16));
    STOCS_CUDA(ctx, ctx->d_cell_start.ensure(starts_cap * 4));
    if (ctx->index_counts_clean < nc1) STOCS_CUDA(ctx, cudaMemsetAsync(counts, 0, nc1 * 4, st));
    ctx->index_counts_clean = 0;   // dirty until this attempt's fill pass has run to completion
    if (S <= (1 << 18)) grid_count_kernel<32><<<(unsigned)(((size_t)S * 32 + 255) / 256), 256, 0, st>>>(ctx->d_spos4.as<float4>(), S, g, r, counts);
    else grid_count_kernel<1><<<nb, 256, 0, st>>>(ctx->d_spos4.as<float4>(), S, g, r, counts);
    cub::DeviceScan::ExclusiveSum(ctx->d_tmp2.p, tmp_bytes, counts, dense_start, (int)nc1, st);
    STOCS_CUDA(ctx, cudaMemcpyAsync(&h_counts[0], dense_start + g.ncells, 4, cudaMemcpyDeviceToHost, st));
    if (S <= (1 << 18)) grid_fill_kernel<32><<<(unsigned)(((size_t)S * 32 + 255) / 256), 256, 0, st>>>(ctx->d_spos4.as<float4>(), S, g, r, dense_start, counts, ctx->d_cand.as<float4>(), (uint32_t)cap);
    else grid_fill_kernel<1><<<nb, 256, 0, st>>>(ctx->d_spos4.as<float4>(), S, g, r, dense_start, counts, ctx->d_cand.as<float4>(), (uint32_t)cap);
    // brick table + compact starts
    STOCS_CUDA(ctx, cudaMemsetAsync(d_occ.p, 0, (size_t)(g.nbricks + 1) * 4, st));
    brick_mask_kernel<<<(unsigned)(((size_t)g.nbricks + 255) / 256), 256, 0, st>>>(dense_start, g.nbricks, d_masks.as<unsigned long long>(),
                                                                                  d_occ.as<uint32_t>(), ctx->d_brick_occ.as<uint32_t>());
    cub::DeviceScan::ExclusiveSum(ctx->d_tmp2.p, tmp_bytes2, d_occ.as<uint32_t>(), d_occ_scan.as<uint32_t>(), (int)(g.nbricks + 1), st);
    STOCS_CUDA(ctx, cudaMemcpyAsync(&h_counts[1], d_occ_scan.as<uint32_t>() + g.nbricks, 4, cudaMemcpyDeviceToHost, st));
    STOCS_CUDA(ctx, cudaMemsetAsync(ctx->d_coarse.p, 0, (size_t)ctx->coarse_words * 4, st));
    brick_table_kernel<<<bb, 128, 0, st>>>(dense_start, d_masks.as<unsigned long long>(), d_occ_scan.as<uint32_t>(), g.nbricks,
                                           dense_start + g.ncells, (uint32_t)starts_cap, ctx->d_bricks.as<uint4>(),
                                           ctx->d_cell_start.as<uint32_t>(), ctx->d_coarse.as<uint32_t>(), g, cshift, cnx + 1, cny + 1);
    STOCS_CUDA(ctx, cudaGetLastError());
    STOCS_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->index_counts_clean = nc1;
    total = h_counts[0]; n_occ = h_counts[1];
    if ((size_t)total <= cap) break;
    if (attempt >= 1) STOCS_FAIL(ctx, STOCS_E_CUDA, "upload_scene: candidate buffer sizing failed");
    cap = (size_t)total + 1024;
  }
  ctx->ncand = total;
  ctx->counters[CTR_OCCUPIED_CELLS] = n_occ;
  tr.mark("index build");
  ctx->counters[CTR_GRID_CELLS] = g.ncells;
  ctx->counters[CTR_CANDIDATES] = total;
  return STOCS_OK;
}

// used by upload_scene in capi.cu
int stocs_pack_scene_attr(stocs_b200_ctx* ctx, const float* d_nrm3, const float* d_cls, int S) {
  STOCS_CUDA(ctx, ctx->d_sattr.ensure((size_t)S * 16));
  pack_attr_kernel<<<(S + 255) / 256, 256, 0, ctx->stream>>>(d_nrm3, d_cls, S, ctx->d_sattr.as<float4>());
  STOCS_CUDA(ctx, cudaGetLastError());
  return STOCS_OK;
}
