// congruent.cu -- congruent-set extraction on the model for a batch of bases.
//
// Replaces stocs_estimator::find_congruent_sets_on_model (reference src/stocs.cpp:753-869) with
// PairCreationFunctor::synch3DContent / getNormalizedEpsilon (pairCreationFunctor.h:96-143) and
// IndexedNormalSet (accelerators/normalset.h:86-122, normalset.hpp:116-131,168-214,
// utils.h:139-148).
//
// The reference inserts the P pairs into a 6-D grid (position cell x 7^3 normal bin) and, for
// every Q pair, rasterises a cone of directions into normal bins of the query's own position
// cell.  A (P,Q) combination is emitted iff
//     cell(P) == cell(Q)  and  normal_bin(P) in cone_bins(Q)  and  |queryQ - invPoint|^2 <= thr
// and the result is ordered by (rank of P in its list, rank of Q in its list).  That predicate
// needs no 6-D grid: one thread computes (cell, normal bin, invPoint) per P entry, a few lanes
// compute (cell, 343-bit cone mask, queryQ) per Q entry, the Q entries are bucketed by a hash of
// (base, cell) -- count, scan, scatter: every bucket a contiguous run of {Q index, cell} records -- and
// one thread per P entry reads the bucket of its own (base, cell), counting, then writing its partners
// in ascending Q rank, which is exactly the std::set order of the reference.  (Round 1 swept the base's whole Q list per P entry: 10^4 x 10^4 on the
// largest base of the YCB frame, 0.12 ms of latency-bound rounds per pose.)
//
// The whole search is ENQUEUED without a host round trip (stocs_congruent_enqueue): list lengths,
// segment offsets and quad counts stay on the device in a StocsPipeState record, the buffers are
// sized by capacities kept in the context, every kernel takes its bounds from the record (grid-stride
// loops), and a search that does not fit raises `overflow` there, which empties its later stages;
// the caller reads the record once, grows the capacities and enqueues the search again.  (Round 1 read
// the list lengths, the quad total and the per-base offsets back one after the other: three
// synchronisations, ~0.2 ms of a 0.45 ms stage on the YCB frame.)
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_radix_sort.cuh>

#include <cfloat>
#include <cmath>

#include "ppf_device.cuh"
#include "stocs_ctx.h"

using namespace stocsm;

PpfView stocs_ppf_view(const stocs_b200_ctx* ctx);

namespace {

struct ModelNorm {   // pairCreationFunctor.h:96-132 + normalset.h:114-122
  float gx, gy, gz;  // bbox centre
  float ratio;       // max extent + 0.001
  float epsilon;     // 1 / egSize
  float nepsilon;    // 1/7 + 1e-5
  int egSize;
};

struct BaseInfo {
  Ppf4 f1, f2;
  float inv1, inv2, cos_alpha;
  uint32_t nP, nQ;
  uint32_t nb_sample;   // directions on the base's cone (normalset.hpp:178-195); table in the cone buffer when <= kConeMax
};
constexpr int kConeMax = 64;   // 2 * ceil(3.5 * 2 pi atan(alpha)) <= 56 for alpha in [0, pi]

__device__ __forceinline__ V3 ld3(const float4* p, int i) { const float4 v = p[i]; return v3(v.x, v.y, v.z); }

// per base: PPF keys of the two base segments, alpha, list lengths
__global__ void cong_count_kernel(const float4* __restrict__ spos4, const float4* __restrict__ sattr, PpfView v,
                                  const int* __restrict__ base_idx4, const float* __restrict__ inv2,
                                  const uint8_t* __restrict__ valid, int n_bases, BaseInfo* __restrict__ info,
                                  float4* __restrict__ cone) {
  const int b = blockIdx.x;
  const int j = threadIdx.x;  // 256 threads: 0..127 -> P bins, 128..255 -> Q bins
  __shared__ BaseInfo s;
  __shared__ uint32_t s_cnt[256];
  if (valid && !valid[b]) {   // a base the sampler rejected keeps its slot with empty lists
    if (j == 0) { BaseInfo z; memset(&z, 0, sizeof(z)); info[b] = z; }
    return;
  }
  if (j == 0) {
    const int* id = base_idx4 + 4 * b;
    const V3 p0 = ld3(spos4, id[0]), p1 = ld3(spos4, id[1]), p2 = ld3(spos4, id[2]), p3 = ld3(spos4, id[3]);
    s.f1 = ppf_compute(p0, ld3(sattr, id[0]), p1, ld3(sattr, id[1]), v.tr, v.rot);
    s.f2 = ppf_compute(p2, ld3(sattr, id[2]), p3, ld3(sattr, id[3]), v.tr, v.rot);
    s.inv1 = inv2[2 * b]; s.inv2 = inv2[2 * b + 1];
    s.cos_alpha = dot(normalized(sub(p1, p0)), normalized(sub(p3, p2)));
  }
  __syncthreads();
  const Ppf4 f = (j < 128) ? s.f1 : s.f2;
  uint32_t c = 0;
  if (!(f.f[0] <= 5 || f.f[1] < 0 || f.f[2] < 0 || f.f[3] < 0)) {
    const uint32_t bin = ppf_source_bin(v, f.f[0] / v.tr, f.f[1] / v.rot, f.f[2] / v.rot, f.f[3] / v.rot, j & 127);
    if (bin != 0xffffffffu) c = v.bin_start[bin + 1] - v.bin_start[bin];
  }
  s_cnt[j] = c;
  __syncthreads();
  if (j == 0) {
    uint32_t nP = 0, nQ = 0;
    for (int k = 0; k < 128; ++k) { nP += s_cnt[k]; nQ += s_cnt[128 + k]; }
    // src/stocs.cpp:788: either list empty => no congruent set
    if (nP == 0 || nQ == 0) { nP = 0; nQ = 0; }
    s.nP = nP; s.nQ = nQ;
  }
  // The cone of directions every Q entry of this base rasterises (normalset.hpp:178-195) is the same
  // set of vectors d0[a] = (sin(alpha) cos(theta_a), sin(alpha) sin(theta_a), cos(alpha)) before the
  // per-entry rotation: computed here once per base instead of once per Q entry (two binary64
  // sin/cos per direction, up to 56 directions, 10^4 entries on some bases)
  float cosAlpha = s.cos_alpha;
  if (cosAlpha > 1.0f) cosAlpha = 1.0f;      // (deviation D2: clamped)
  if (cosAlpha < -1.0f) cosAlpha = -1.0f;
  const float alpha = acos_f(cosAlpha);
  const float perimeter = (float)((double)2.0f * kPi * (double)atan_f(alpha));
  const unsigned nbSample = (unsigned)(2.0f * ceilf(perimeter * 7.0f / 2.0f));
  if ((unsigned)j < nbSample && j < kConeMax) {
    const float angleStep = (float)((double)2.0f * kPi / (double)(float)nbSample);
    const float sinAlpha = sin_f(alpha);
    const float theta = (float)j * angleStep;
    cone[(size_t)b * kConeMax + j] = make_float4(sinAlpha * cos_f(theta), sinAlpha * sin_f(theta), cosAlpha, 0.f);
  }
  if (j == 0) { s.nb_sample = nbSample; info[b] = s; }
}

// exclusive scan of one value per thread over a 256-thread block; *total = the block's sum
__device__ __forceinline__ unsigned long long block_excl_scan_256(unsigned long long v, unsigned long long* s_buf,
                                                                  unsigned long long* total) {
  const int j = threadIdx.x;
  s_buf[j] = v;
  __syncthreads();
  for (int o = 1; o < 256; o <<= 1) {
    const unsigned long long up = (j >= o) ? s_buf[j - o] : 0ull;
    __syncthreads();
    s_buf[j] += up;
    __syncthreads();
  }
  const unsigned long long incl = s_buf[j];
  *total = s_buf[255];
  __syncthreads();
  return incl - v;
}

// segment offsets of the flat code buffer, [P_0..P_{n-1} | Q_0..Q_{n-1} | total], from the list lengths
// (index bookkeeping only; one block).  Lists that do not fit the code buffers leave every segment
// empty and raise the overflow flag.
__global__ void __launch_bounds__(256) cong_seg_kernel(const BaseInfo* __restrict__ info, int n_bases, uint32_t* __restrict__ seg,
                                                        unsigned long long cap_codes, StocsPipeState* __restrict__ stt) {
  __shared__ unsigned long long s_buf[256];
  const int j = threadIdx.x;
  const int per = (n_bases + 255) / 256;
  const int b0 = min(n_bases, j * per), b1 = min(n_bases, b0 + per);
  unsigned long long locP = 0, locQ = 0;
  for (int b = b0; b < b1; ++b) { locP += info[b].nP; locQ += info[b].nQ; }
  unsigned long long totalP, totalQ;
  unsigned long long offP = block_excl_scan_256(locP, s_buf, &totalP);
  unsigned long long offQ = block_excl_scan_256(locQ, s_buf, &totalQ);
  const unsigned long long total = totalP + totalQ;
  // (2^28 entries: the prepare kernel numbers 8 work items per Q entry in 32 bits)
  const uint32_t ovf = (total >= (1ull << 28)) ? 4u : (total > cap_codes ? 1u : 0u);
  if (ovf) {
    for (int b = b0; b < b1; ++b) { seg[b] = 0u; seg[n_bases + b] = 0u; }
  } else {
    offQ += totalP;
    for (int b = b0; b < b1; ++b) {
      seg[b] = (uint32_t)offP; offP += info[b].nP;
      seg[n_bases + b] = (uint32_t)offQ; offQ += info[b].nQ;
    }
  }
  if (j == 0) {
    seg[2 * n_bases] = ovf ? 0u : (uint32_t)total;
    stt->need_codes = total;
    stt->totalP = ovf ? 0u : (uint32_t)totalP;
    stt->total = ovf ? 0u : (uint32_t)total;
    stt->overflow |= ovf;
  }
}

// copy the source-bin ranges of both lists into the flat code buffer (unsorted): the block walks the
// base's nP + nQ entries as one flat range and finds each entry's source bin by binary search over the
// bins' output offsets (one bin after the other cost 256 dependent little loops: 61 us per 100 bases)
__global__ void __launch_bounds__(256) cong_gather_kernel(PpfView v, const BaseInfo* __restrict__ info, const uint32_t* __restrict__ seg_off,
                                                           int n_bases, uint32_t* __restrict__ codes, const StocsPipeState* __restrict__ stt) {
  const int b = blockIdx.x;
  const int j = threadIdx.x;
  __shared__ uint32_t s_start[256], s_loc[257];   // s_loc: exclusive offsets of the 256 bins inside the base's flat range
  __shared__ unsigned long long s_buf[256];
  if (stt->overflow) return;
  const BaseInfo bi = info[b];
  if (bi.nP == 0) return;
  const Ppf4 f = (j < 128) ? bi.f1 : bi.f2;
  uint32_t st = 0, c = 0;
  const uint32_t bin = ppf_source_bin(v, f.f[0] / v.tr, f.f[1] / v.rot, f.f[2] / v.rot, f.f[3] / v.rot, j & 127);
  if (bin != 0xffffffffu) { st = v.bin_start[bin]; c = v.bin_start[bin + 1] - st; }
  s_start[j] = st;
  unsigned long long total;
  s_loc[j] = (uint32_t)block_excl_scan_256((unsigned long long)c, s_buf, &total);
  if (j == 0) s_loc[256] = (uint32_t)total;
  __syncthreads();
  const uint32_t n = bi.nP + bi.nQ;       // == total (bins 0..127 hold the P list, 128..255 the Q list)
  const uint32_t outP = seg_off[b], outQ = seg_off[n_bases + b];
  // gridDim.y blocks share a base (a few bases carry lists of 10^4 entries: one block each was the stage's tail)
  for (uint32_t e = blockIdx.y * 256 + j; e < n; e += 256 * gridDim.y) {
    int lo = 0, hi = 256;                 // last bin whose offset is <= e (empty bins share offsets: the last one is the non-empty one)
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (s_loc[mid] <= e) lo = mid; else hi = mid; }
    const uint32_t code = v.pairs[s_start[lo] + (e - s_loc[lo])];
    codes[(e < bi.nP) ? (outP + e) : (outQ + (e - bi.nP))] = code;
  }
}

__device__ __forceinline__ int index_normal(const ModelNorm& mn, V3 n) {
  const float cx = (n.x / 2.0f + 0.5f) / mn.nepsilon, cy = (n.y / 2.0f + 0.5f) / mn.nepsilon,
              cz = (n.z / 2.0f + 0.5f) / mn.nepsilon;
  return (int)cz * 49 + ((int)cy * 7 + (int)cx);
}
__device__ __forceinline__ int index_pos(const ModelNorm& mn, V3 p) {
  const V3 c = divs(p, mn.epsilon);
  return (int)c.z * mn.egSize * mn.egSize + ((int)c.y * mn.egSize + (int)c.x);
}
__device__ __forceinline__ V3 to_unit(const ModelNorm& mn, V3 p) {
  const V3 d = divs(sub(p, v3(mn.gx, mn.gy, mn.gz)), mn.ratio);
  return v3(d.x + 0.5f, d.y + 0.5f, d.z + 0.5f);
}

struct PEntry { float ix, iy, iz; int cell; int nbin; int base; };   // invPoint (model frame)
// Q entries are bucketed by (base, position cell) in one table of `table_size` (a power of two, at least
// twice the code capacity) buckets; a bucket may mix entries of different bases and cells, told apart on the read
constexpr uint32_t kNoEntry = 0xffffffffu;
__device__ __forceinline__ uint32_t bucket_of(int b, int cell, int table_bits) {
  return (((uint32_t)cell * 2654435761u) ^ ((uint32_t)b * 0x9E3779B1u + 0x7F4A7C15u)) >> (32 - table_bits);
}
struct QEntry { float qx, qy, qz; uint32_t mask[11]; };          // queryQ (model frame), cone bins

// entry e of the flat (sorted) code buffer: P entries first, then Q entries
__global__ void cong_prepare_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ seg_off,
                                    const BaseInfo* __restrict__ info, int n_bases, const StocsPipeState* __restrict__ stt,
                                    const float4* __restrict__ mpos4, ModelNorm mn, PEntry* __restrict__ pe,
                                    QEntry* __restrict__ qe, int* __restrict__ qcell, uint32_t* __restrict__ bcount,
                                    uint32_t* __restrict__ qslot, int table_bits, const float4* __restrict__ cone) {
  // Work items: one thread per P entry, then -- from the next multiple of 32, so that a warp never mixes
  // the two kinds -- kQLanes consecutive lanes per Q entry, which share the entry's cone of up to 56
  // directions (the serial loop over the cone was the stage's critical path) and OR their bin masks.
  constexpr uint32_t kQLanes = 8;
  const uint32_t totalP = stt->totalP, total = stt->total;
  const uint32_t P32 = (totalP + 31u) & ~31u;
  const uint32_t items = P32 + (total - totalP) * kQLanes;
  const uint32_t items32 = (items + 31u) & ~31u;
  for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < items32; v += gridDim.x * blockDim.x) {
  const bool isP = v < totalP;
  const bool inQ = v >= P32;                       // warp-uniform
  const uint32_t ql = inQ ? ((v - P32) % kQLanes) : 0u;   // lane of the Q entry's group
  const uint32_t e = isP ? v : (inQ ? totalP + (v - P32) / kQLanes : total);
  const bool live = e < total;
  QEntry o;
  for (int k = 0; k < 11; ++k) o.mask[k] = 0u;
  o.qx = o.qy = o.qz = 0.f;
  int b = 0, qc = 0;
  if (live) {
  // find the base (segment) by binary search in seg_off (2*n_bases+1 entries)
  int lo = isP ? 0 : n_bases, hi = isP ? n_bases : 2 * n_bases;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (seg_off[mid] <= e) lo = mid; else hi = mid;
  }
  b = isP ? lo : lo - n_bases;
  const BaseInfo bi = info[b];
  const uint32_t code = codes[e];
  const int i1 = (int)(code >> 16), i2 = (int)(code & 0xffffu);
  const V3 w1 = ld3(mpos4, i1), w2 = ld3(mpos4, i2);
  const V3 u1 = to_unit(mn, w1), u2 = to_unit(mn, w2);
  const V3 du = sub(u2, u1);
  const V3 dirn = normalized(du);
  if (isP) {
    PEntry po;
    const V3 pos = add(u1, scale(du, bi.inv1));
    po.cell = index_pos(mn, pos);
    po.nbin = index_normal(mn, dirn);
    const V3 ip = add(w1, scale(sub(w2, w1), bi.inv1));
    po.ix = ip.x; po.iy = ip.y; po.iz = ip.z;
    po.base = b;
    pe[e] = po;
  } else {
    const V3 query = add(u1, scale(du, bi.inv2));
    const V3 qq = add(w1, scale(sub(w2, w1), bi.inv2));
    o.qx = qq.x; o.qy = qq.y; o.qz = qq.z;
    qc = index_pos(mn, query);
    // normalset.hpp:178-195 (cosAlpha clamped: deviation D2); the unrotated cone comes from the base's table
    const unsigned nbSample = bi.nb_sample;
    const bool tabled = nbSample <= (unsigned)kConeMax;
    float cosAlpha = bi.cos_alpha;
    if (cosAlpha > 1.0f) cosAlpha = 1.0f;
    if (cosAlpha < -1.0f) cosAlpha = -1.0f;
    float angleStep = 0.f, sinAlpha = 0.f;
    if (!tabled) {   // (cannot happen for alpha in [0, pi]; kept so that the result never depends on the table size)
      const float alpha = acos_f(cosAlpha);
      angleStep = (float)((double)2.0f * kPi / (double)(float)nbSample);
      sinAlpha = sin_f(alpha);
    }
    // Quaternion::setFromTwoVectors((0,0,1), dirn)  (deviation D5 on the antiparallel branch)
    const V3 v0 = v3(0.f, 0.f, 1.f);
    const V3 v1 = normalized(dirn);
    float c = dot(v1, v0);
    V3 qv; float qw;
    if (c < -1.0f + 1e-5f) {
      c = c > -1.0f ? c : -1.0f;
      V3 ax = cross(v0, v1);
      if (sqnorm(ax) > 0.0f) ax = normalized(ax); else ax = v3(1.f, 0.f, 0.f);
      const float w2q = (1.0f + c) * 0.5f;
      qw = sqrtf(w2q);
      qv = scale(ax, sqrtf(1.0f - w2q));
    } else {
      const V3 axis = cross(v0, v1);
      const float s = sqrtf((1.0f + c) * 2.0f);
      const float invs = 1.0f / s;
      qv = scale(axis, invs);
      qw = s * 0.5f;
    }
    for (unsigned a = ql; a < nbSample; a += kQLanes) {
      V3 d0;
      if (tabled) {
        const float4 t = cone[(size_t)b * kConeMax + a];
        d0 = v3(t.x, t.y, t.z);
      } else {
        const float theta = (float)a * angleStep;
        d0 = v3(sinAlpha * cos_f(theta), sinAlpha * sin_f(theta), cosAlpha);
      }
      V3 uv = cross(qv, d0);
      uv = add(uv, uv);
      const V3 rot = add(add(d0, scale(uv, qw)), cross(qv, uv));
      const int id = index_normal(mn, normalized(rot));
      if (id >= 0 && id < 343) o.mask[id >> 5] |= 1u << (id & 31);
    }
  }
  }
  if (inQ) {   // whole warp: OR the bin masks of the kQLanes lanes of each entry
#pragma unroll
    for (int k = 0; k < 11; ++k) {
      uint32_t m = o.mask[k];
      m |= __shfl_xor_sync(0xffffffffu, m, 1);
      m |= __shfl_xor_sync(0xffffffffu, m, 2);
      m |= __shfl_xor_sync(0xffffffffu, m, 4);
      o.mask[k] = m;
    }
    if (live && ql == 0) {
      qe[e - totalP] = o;
      qcell[e - totalP] = qc;
      const uint32_t h = bucket_of(b, qc, table_bits);
      qslot[e - totalP] = h;
      atomicAdd(&bcount[h], 1u);
    }
  }
  }
}

// second half of the bucketing: every Q entry takes a slot of its bucket, from the back (the counts go
// back to zero, so the table needs no clearing between searches)
__global__ void cong_scatter_kernel(const StocsPipeState* __restrict__ stt, const uint32_t* __restrict__ qslot,
                                    const int* __restrict__ qcell, const uint32_t* __restrict__ bstart,
                                    uint32_t* __restrict__ bcount, uint2* __restrict__ bucket) {
  const uint32_t totalQ = stt->total - stt->totalP;
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < totalQ; q += gridDim.x * blockDim.x) {
    const uint32_t h = qslot[q];
    const uint32_t pos = bstart[h] + atomicSub(&bcount[h], 1u) - 1u;
    bucket[pos] = make_uint2(q, (uint32_t)qcell[q]);
  }
}

// does Q entry q (index into the Q block, same base and cell as p) form a congruent set with P entry p?
__device__ __forceinline__ bool congruent_pair(const PEntry& p, const QEntry* __restrict__ qe, uint32_t q, float thr) {
  const QEntry& e = qe[q];
  if (!((e.mask[p.nbin >> 5] >> (p.nbin & 31)) & 1u)) return false;
  const float dx = e.qx - p.ix, dy = e.qy - p.iy, dz = e.qz - p.iz;
  return (dx * dx + (dy * dy + dz * dz)) <= thr;  // squared distance vs UNSQUARED threshold (quirk 1)
}

// one warp per P entry, 32 records of its bucket per step; WRITE=false counts its partners, WRITE=true
// emits the quads in ascending Q rank.  (One THREAD per P entry left the stage waiting on the few hundred
// entries whose cell holds a thousand Q entries: 64 + 93 us on a YCB frame with one 10^4-entry base.)
template <bool WRITE>
__global__ void __launch_bounds__(256) cong_match_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ seg_off,
                                  int n_bases, const StocsPipeState* __restrict__ stt, const PEntry* __restrict__ pe,
                                  const QEntry* __restrict__ qe, float thr,
                                  uint32_t* __restrict__ counts, const uint32_t* __restrict__ out_off,
                                  int* __restrict__ quads, const uint32_t* __restrict__ bstart,
                                  const uint2* __restrict__ bucket, int table_bits) {
  constexpr uint32_t kLocal = 64;
  __shared__ uint32_t s_found[8][kLocal];
  const uint32_t totalP = stt->totalP;
  if (WRITE && stt->overflow) return;   // the quads would not fit: the caller grows the buffer and searches again
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const unsigned lt = (1u << lane) - 1u;
  const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; wid < totalP; wid += nwarps) {
    uint32_t o0 = 0, want = 0;
    if (WRITE) {
      o0 = out_off[wid]; want = out_off[wid + 1] - o0;
      if (want == 0) continue;
    }
    const PEntry p = pe[wid];
    if (p.nbin < 0 || p.nbin >= 343) { if (!WRITE && lane == 0) counts[wid] = 0u; continue; }  // std::array::at would throw
    const uint32_t q0 = seg_off[n_bases + p.base] - totalP, q1 = seg_off[n_bases + p.base + 1] - totalP;
    const uint32_t h = bucket_of(p.base, p.cell, table_bits);
    const uint32_t r0 = bstart[h], r1 = bstart[h + 1];
    const uint32_t pcell = (uint32_t)p.cell;
    // a record of the bucket is a partner when it is a Q entry of this base in this cell (the bucket may
    // hold others) and passes the normal-bin and distance tests (the 56-byte Q entry is read only then)
    auto partner = [&](uint32_t r, uint32_t& q) -> bool {
      if (r >= r1) return false;
      const uint2 rec = bucket[r];
      q = rec.x;
      return q >= q0 && q < q1 && rec.y == pcell && congruent_pair(p, qe, q, thr);
    };
    if (!WRITE) {
      uint32_t cnt = 0;
      for (uint32_t r = r0; r < r1; r += 32) {
        uint32_t q;
        cnt += __popc(__ballot_sync(0xffffffffu, partner(r + lane, q)));
      }
      if (lane == 0) counts[wid] = cnt;
    } else {
      // partners in ascending Q rank; a bucket holds its records in arrival (arbitrary) order
      const uint32_t pcode = codes[wid];
      if (want <= kLocal) {   // collect, then every partner counts the smaller ones: that is its place
        uint32_t n = 0;
        for (uint32_t r = r0; r < r1; r += 32) {
          uint32_t q = 0;
          const bool m = partner(r + lane, q);
          const unsigned bal = __ballot_sync(0xffffffffu, m);
          if (m) s_found[w][n + __popc(bal & lt)] = q;
          n += __popc(bal);
        }
        __syncwarp();
        for (uint32_t k = lane; k < n; k += 32) {
          const uint32_t q = s_found[w][k];
          uint32_t rank = 0;
          for (uint32_t j = 0; j < n; ++j) rank += (s_found[w][j] < q) ? 1u : 0u;
          const uint32_t qcode = codes[totalP + q];
          reinterpret_cast<int4*>(quads)[o0 + rank] = make_int4((int)(pcode >> 16), (int)(pcode & 0xffffu), (int)(qcode >> 16), (int)(qcode & 0xffffu));
        }
        __syncwarp();
      } else {                // many partners: the smallest rank above the previous one, `want` times
        uint32_t last = 0; bool have_last = false;
        for (uint32_t k = 0; k < want; ++k) {
          uint32_t best = kNoEntry;
          for (uint32_t r = r0; r < r1; r += 32) {
            uint32_t q = 0;
            if (partner(r + lane, q) && q < best && (!have_last || q > last)) best = q;
          }
          best = __reduce_min_sync(0xffffffffu, best);
          last = best; have_last = true;
          if (lane == 0) {
            const uint32_t qcode = codes[totalP + best];
            reinterpret_cast<int4*>(quads)[o0 + k] = make_int4((int)(pcode >> 16), (int)(pcode & 0xffffu), (int)(qcode >> 16), (int)(qcode & 0xffffu));
          }
        }
      }
    }
  }
}

// quad total and per-base quad offsets from the scanned per-P counts (one block)
__global__ void __launch_bounds__(256) cong_base_offsets_kernel(const uint32_t* __restrict__ seg_off, const uint32_t* __restrict__ pscan,
                                                                 int n_bases, unsigned long long cap_quads,
                                                                 StocsPipeState* __restrict__ stt, long long* __restrict__ quad_off) {
  const uint32_t totalP = stt->totalP;
  const uint32_t total_quads = pscan[totalP];
  const bool ovf = (unsigned long long)total_quads > cap_quads;
  for (int b = threadIdx.x; b <= n_bases; b += blockDim.x) {
    const uint32_t e = (b < n_bases) ? seg_off[b] : totalP;
    quad_off[b] = ovf ? 0ll : ((e < totalP) ? (long long)pscan[e] : (long long)total_quads);
  }
  if (threadIdx.x == 0) {
    stt->need_quads = total_quads;
    stt->total_quads = ovf ? 0u : total_quads;
    if (ovf) stt->overflow |= 2u;
  }
}

}  // namespace

// Derives the unit-cube normalisation of the model (host scalars; exact IEEE ops, same as the
// device would do) -- pairCreationFunctor.h:96-132, normalset.h:114-122.
static ModelNorm model_norm(const stocs_b200_ctx* ctx) {
  const float big = FLT_MAX / 2;
  float mn[3] = {big, big, big}, mx[3] = {-big, -big, -big};
  for (int i = 0; i < ctx->M; ++i)
    for (int k = 0; k < 3; ++k) {
      const float c = ctx->h_mpos[3 * (size_t)i + k];
      if (c < mn[k]) mn[k] = c;
      if (c > mx[k]) mx[k] = c;
    }
  ModelNorm m;
  const float ex = mx[0] - mn[0], ey = mx[1] - mn[1], ez = mx[2] - mn[2];
  m.gx = mn[0] + (ex / 2.0f); m.gy = mn[1] + (ey / 2.0f); m.gz = mn[2] + (ez / 2.0f);
  const double r = std::max((double)ez + 0.001, std::max((double)ey + 0.001, (double)ex + 0.001));
  m.ratio = (float)r;
  const float eps = ctx->eps / m.ratio;
  const int gridDepth = (int)(-stocsm::log2_f(eps));
  m.egSize = 1 << (gridDepth < 0 ? 0 : (gridDepth > 10 ? 10 : gridDepth));
  m.epsilon = 1.f / (float)m.egSize;
  m.nepsilon = (float)((double)(1.0f / 7.0f) + 0.00001);
  return m;
}

// Enqueues the congruent-set search of n_bases bases on `st`; nothing is read back.
//   d_base_idx4 / d_inv2 / d_valid (may be NULL: all valid): per base, on the device
//   d_state: the run's StocsPipeState (the CALLER zeroes it); this search fills need_codes, need_quads,
//            totalP, total, total_quads and may raise overflow bits 1 / 2 / 4
//   d_quad_off: n_bases + 1 offsets into the quad buffer ctx->pool[POOL_CONG_QUADS]
// Sizes of one congruent-set search against the context's capacities.
struct CongSizes { size_t cap, capq, table_size; int table_bits, end_bit; size_t tb, tb2, tb3; };

#define CG(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) { ctx->err = std::string(#call) + ": " + cudaGetErrorString(_e); return STOCS_E_CUDA; } } while (0)
// Grows every buffer of a search over n_bases bases; enqueues nothing.
static int cong_reserve(stocs_b200_ctx* ctx, int n_bases, CongSizes& z) {
  cudaStream_t st = ctx->stream;   // (the cub size queries below enqueue nothing)
  DevBuf &d_info = ctx->pool[POOL_CONG_INFO], &d_seg = ctx->pool[POOL_CONG_SEG], &d_codes_a = ctx->pool[POOL_CONG_CODES_A], &d_codes_b = ctx->pool[POOL_CONG_CODES_B], &d_tmp = ctx->pool[POOL_CONG_TMP],
         &d_pe = ctx->pool[POOL_CONG_PE], &d_qe = ctx->pool[POOL_CONG_QE], &d_qcell = ctx->pool[POOL_CONG_QCELL], &d_cnt = ctx->pool[POOL_CONG_CNT], &d_scan = ctx->pool[POOL_CONG_SCAN],
         &quads_buf = ctx->pool[POOL_CONG_QUADS], &d_bcount = ctx->pool[POOL_CONG_HEAD], &d_cone = ctx->pool[POOL_CONG_CONE],
         &d_qslot = ctx->pool[POOL_CONG_NEXT], &d_bstart = ctx->pool[POOL_CONG_BSTART], &d_bucket = ctx->pool[POOL_CONG_BUCKET];
  const size_t cap = (size_t)ctx->cong_cap_codes, capq = (size_t)ctx->cong_cap_quads;
  z.cap = cap; z.capq = capq;
  CG(d_info.ensure((size_t)n_bases * sizeof(BaseInfo)));
  CG(d_seg.ensure(((size_t)2 * n_bases + 1) * 4));
  CG(d_codes_a.ensure(cap * 4));
  CG(d_codes_b.ensure(cap * 4));
  CG(d_pe.ensure(cap * sizeof(PEntry)));
  CG(d_qe.ensure(cap * sizeof(QEntry)));
  CG(d_qcell.ensure(cap * 4));
  CG(d_cnt.ensure((cap + 1) * 4));
  CG(d_scan.ensure((cap + 1) * 4));
  CG(quads_buf.ensure(capq * 16));
  int table_bits = 10;
  while (table_bits < 31 && ((size_t)1 << table_bits) < 2 * cap) ++table_bits;
  const size_t table_size = (size_t)1 << table_bits;
  z.table_bits = table_bits; z.table_size = table_size;
  if (d_bcount.bytes < (table_size + 1) * 4) ctx->cong_bcount_clean = false;   // a new buffer holds no zeroed counters
  CG(d_bcount.ensure((table_size + 1) * 4));
  CG(d_bstart.ensure((table_size + 1) * 4));
  CG(d_bucket.ensure(cap * 8));
  CG(d_cone.ensure((size_t)n_bases * kConeMax * 16));
  CG(d_qslot.ensure(cap * 4));
  // (id1 << 16) | id2 with ids < M: the bits above 16 + ceil(log2 M) are zero
  int end_bit = 17;
  while (end_bit < 32 && (1 << (end_bit - 16)) < ctx->M) ++end_bit;
  z.end_bit = end_bit;
  size_t tb = 0, tb2 = 0, tb3 = 0;
  cub::DeviceSegmentedRadixSort::SortKeys(nullptr, tb, d_codes_a.as<uint32_t>(), d_codes_b.as<uint32_t>(), (int)cap,
                                          2 * n_bases, d_seg.as<uint32_t>(), d_seg.as<uint32_t>() + 1, 0, end_bit, st);
  cub::DeviceScan::ExclusiveSum(nullptr, tb2, d_cnt.as<uint32_t>(), d_scan.as<uint32_t>(), (int)(cap + 1), st);
  cub::DeviceScan::ExclusiveSum(nullptr, tb3, d_bcount.as<uint32_t>(), d_bstart.as<uint32_t>(), (int)(table_size + 1), st);
  CG(d_tmp.ensure(std::max(tb, std::max(tb2, tb3))));
  z.tb = tb; z.tb2 = tb2; z.tb3 = tb3;
  return STOCS_OK;
}

int stocs_congruent_reserve(stocs_b200_ctx* ctx, int n_bases) {
  CongSizes z;
  return n_bases > 0 ? cong_reserve(ctx, n_bases, z) : STOCS_OK;
}

// Buffers are sized by ctx->cong_cap_codes / cong_cap_quads; stocs_congruent_grow() raises them from a
// state record that came back with overflow set.
int stocs_congruent_enqueue(stocs_b200_ctx* ctx, int n_bases, const int* d_base_idx4, const float* d_inv2,
                            const uint8_t* d_valid, StocsPipeState* d_state, long long* d_quad_off, cudaStream_t st) {
  if (n_bases <= 0) return STOCS_OK;
  const PpfView v = stocs_ppf_view(ctx);
  DevBuf &d_info = ctx->pool[POOL_CONG_INFO], &d_seg = ctx->pool[POOL_CONG_SEG], &d_codes_a = ctx->pool[POOL_CONG_CODES_A], &d_codes_b = ctx->pool[POOL_CONG_CODES_B], &d_tmp = ctx->pool[POOL_CONG_TMP],
         &d_pe = ctx->pool[POOL_CONG_PE], &d_qe = ctx->pool[POOL_CONG_QE], &d_qcell = ctx->pool[POOL_CONG_QCELL], &d_cnt = ctx->pool[POOL_CONG_CNT], &d_scan = ctx->pool[POOL_CONG_SCAN],
         &quads_buf = ctx->pool[POOL_CONG_QUADS], &d_bcount = ctx->pool[POOL_CONG_HEAD], &d_cone = ctx->pool[POOL_CONG_CONE],
         &d_qslot = ctx->pool[POOL_CONG_NEXT], &d_bstart = ctx->pool[POOL_CONG_BSTART], &d_bucket = ctx->pool[POOL_CONG_BUCKET];
  CongSizes z;
  if (const int rc = cong_reserve(ctx, n_bases, z)) return rc;
  const size_t cap = z.cap, capq = z.capq, table_size = z.table_size;
  size_t tb = z.tb, tb2 = z.tb2, tb3 = z.tb3;   // (cub takes them by reference)
  const int table_bits = z.table_bits, end_bit = z.end_bit;
  // bucket counters: every search leaves them zero (cong_scatter_kernel), so they are cleared only when
  // the buffer is new -- or after a search that did not run to its end
  const bool fresh = ctx->cong_table_size != (long long)table_size || !ctx->cong_bcount_clean;
  if (fresh) CG(cudaMemsetAsync(d_bcount.p, 0, (table_size + 1) * 4, st));
  ctx->cong_table_size = (long long)table_size;
  ctx->cong_bcount_clean = false;   // until the whole search has been enqueued

  cong_count_kernel<<<n_bases, 256, 0, st>>>(ctx->d_spos4.as<float4>(), ctx->d_sattr.as<float4>(), v, d_base_idx4, d_inv2,
                                             d_valid, n_bases, d_info.as<BaseInfo>(), d_cone.as<float4>());
  cong_seg_kernel<<<1, 256, 0, st>>>(d_info.as<BaseInfo>(), n_bases, d_seg.as<uint32_t>(), (unsigned long long)cap, d_state);
  cong_gather_kernel<<<dim3((unsigned)n_bases, 8), 256, 0, st>>>(v, d_info.as<BaseInfo>(), d_seg.as<uint32_t>(), n_bases, d_codes_a.as<uint32_t>(), d_state);
  // per-list sort by (id1, id2): the reference's list order (insertion order of the pair loop).
  // num_items only sizes the library's scratch; the segments come from d_seg on the device.
  cub::DeviceSegmentedRadixSort::SortKeys(d_tmp.p, tb, d_codes_a.as<uint32_t>(), d_codes_b.as<uint32_t>(), (int)cap,
                                          2 * n_bases, d_seg.as<uint32_t>(), d_seg.as<uint32_t>() + 1, 0, end_bit, st);
  const uint32_t* codes = d_codes_b.as<uint32_t>();
  const ModelNorm mn = model_norm(ctx);
  const unsigned wide = (unsigned)ctx->num_sms * 8;

  cong_prepare_kernel<<<wide, 128, 0, st>>>(codes, d_seg.as<uint32_t>(), d_info.as<BaseInfo>(), n_bases, d_state,
                                            ctx->d_mpos4.as<float4>(), mn, d_pe.as<PEntry>(), d_qe.as<QEntry>(), d_qcell.as<int>(),
                                            d_bcount.as<uint32_t>(), d_qslot.as<uint32_t>(), table_bits, d_cone.as<float4>());
  cub::DeviceScan::ExclusiveSum(d_tmp.p, tb3, d_bcount.as<uint32_t>(), d_bstart.as<uint32_t>(), (int)(table_size + 1), st);
  cong_scatter_kernel<<<wide, 256, 0, st>>>(d_state, d_qslot.as<uint32_t>(), d_qcell.as<int>(), d_bstart.as<uint32_t>(),
                                            d_bcount.as<uint32_t>(), d_bucket.as<uint2>());
  CG(cudaMemsetAsync(d_cnt.p, 0, (cap + 1) * 4, st));
  const unsigned mgrid = (unsigned)ctx->num_sms * 4;   // one wave of 256-thread blocks at up to 64 registers; one P entry per warp at a time
  cong_match_kernel<false><<<mgrid, 256, 0, st>>>(codes, d_seg.as<uint32_t>(), n_bases, d_state, d_pe.as<PEntry>(),
                                                  d_qe.as<QEntry>(), ctx->eps, d_cnt.as<uint32_t>(), nullptr, nullptr,
                                                  d_bstart.as<uint32_t>(), d_bucket.as<uint2>(), table_bits);
  cub::DeviceScan::ExclusiveSum(d_tmp.p, tb2, d_cnt.as<uint32_t>(), d_scan.as<uint32_t>(), (int)(cap + 1), st);
  cong_base_offsets_kernel<<<1, 256, 0, st>>>(d_seg.as<uint32_t>(), d_scan.as<uint32_t>(), n_bases, (unsigned long long)capq,
                                              d_state, d_quad_off);
  cong_match_kernel<true><<<mgrid, 256, 0, st>>>(codes, d_seg.as<uint32_t>(), n_bases, d_state, d_pe.as<PEntry>(),
                                                 d_qe.as<QEntry>(), ctx->eps, nullptr, d_scan.as<uint32_t>(),
                                                 quads_buf.as<int>(), d_bstart.as<uint32_t>(), d_bucket.as<uint2>(), table_bits);
  CG(cudaGetLastError());
  ctx->cong_bcount_clean = true;
#undef CG
  return STOCS_OK;
}

// After a state record came back with overflow bits 1 or 2: raise the capacities to what the search
// needs (+25 %).  Returns false when the search can never fit (bit 4: pair lists of 2^28 entries or more).
bool stocs_congruent_grow(stocs_b200_ctx* ctx, const StocsPipeState& s) {
  if (s.overflow & 4u) return false;
  if ((s.overflow & 1u) && (long long)s.need_codes > ctx->cong_cap_codes) {
    long long want = (long long)(s.need_codes + s.need_codes / 4 + 1024);
    if (want >= (1ll << 28)) want = (1ll << 28) - 1;
    ctx->cong_cap_codes = want;
  }
  if ((s.overflow & 2u) && (long long)s.need_quads > ctx->cong_cap_quads)
    ctx->cong_cap_quads = (long long)(s.need_quads + s.need_quads / 4 + 1024);
  return true;
}

extern "C" int stocs_b200_find_congruent(stocs_b200_ctx* ctx, int n_bases, const int32_t* base_idx4, const float* inv2,
                                         int32_t* quads4, int64_t cap, int64_t* quad_offsets) {
  if (!ctx) return STOCS_E_ARG;
  if (ctx->S <= 0 || ctx->M <= 0) STOCS_FAIL(ctx, STOCS_E_STATE, "find_congruent: upload_model and upload_scene first");
  if (n_bases < 0 || !quad_offsets || cap < 0 || (n_bases > 0 && (!base_idx4 || !inv2)))
    STOCS_FAIL(ctx, STOCS_E_ARG, "find_congruent: bad argument");
  for (int i = 0; i < 4 * n_bases; ++i)
    if (base_idx4[i] < 0 || base_idx4[i] >= ctx->S) STOCS_FAIL(ctx, STOCS_E_ARG, "find_congruent: base index out of range");
  quad_offsets[0] = 0;
  if (n_bases == 0) return STOCS_OK;
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  STOCS_CUDA(ctx, ctx->d_tmp2.ensure((size_t)n_bases * 24));
  int* d_ids = ctx->d_tmp2.as<int>();
  float* d_inv = (float*)(d_ids + 4 * (size_t)n_bases);
  STOCS_CUDA(ctx, cudaMemcpyAsync(d_ids, base_idx4, (size_t)n_bases * 16, cudaMemcpyHostToDevice, st));
  STOCS_CUDA(ctx, cudaMemcpyAsync(d_inv, inv2, (size_t)n_bases * 8, cudaMemcpyHostToDevice, st));
  STOCS_CUDA(ctx, ctx->pool[POOL_PIPE_STATE].ensure(sizeof(StocsPipeState)));
  STOCS_CUDA(ctx, ctx->pool[POOL_CONG_QOFF].ensure((size_t)(n_bases + 1) * 8));
  StocsPipeState* d_state = ctx->pool[POOL_PIPE_STATE].as<StocsPipeState>();
  long long* d_qoff = ctx->pool[POOL_CONG_QOFF].as<long long>();
  StocsPipeState& hs = *ctx->h_pipe_state;
  for (int attempt = 0;; ++attempt) {
    STOCS_CUDA(ctx, cudaMemsetAsync(d_state, 0, sizeof(StocsPipeState), st));
    const int rc = stocs_congruent_enqueue(ctx, n_bases, d_ids, d_inv, nullptr, d_state, d_qoff, st);
    if (rc) return rc;
    STOCS_CUDA(ctx, cudaMemcpyAsync(&hs, d_state, sizeof(StocsPipeState), cudaMemcpyDeviceToHost, st));
    STOCS_CUDA(ctx, cudaMemcpyAsync(quad_offsets, d_qoff, (size_t)(n_bases + 1) * 8, cudaMemcpyDeviceToHost, st));
    STOCS_CUDA(ctx, cudaStreamSynchronize(st));
    if (!hs.overflow) break;
    if (!stocs_congruent_grow(ctx, hs) || attempt >= 2) STOCS_FAIL(ctx, STOCS_E_ARG, "find_congruent: pair lists too long");
  }
  const long long total = (long long)hs.total_quads;
  if (total > cap) STOCS_FAIL(ctx, STOCS_E_CAPACITY, "find_congruent: quads4 capacity too small");
  if (total > 0) {
    if (!quads4) STOCS_FAIL(ctx, STOCS_E_ARG, "find_congruent: quads4 is NULL");
    STOCS_CUDA(ctx, cudaMemcpyAsync(quads4, ctx->pool[POOL_CONG_QUADS].p, (size_t)total * 16, cudaMemcpyDeviceToHost, st));
    STOCS_CUDA(ctx, cudaStreamSynchronize(st));
  }
  return STOCS_OK;
}
