// k_index.cuh -- K4: the flat device-resident spatial index that replaces nanoflann's
// KD-tree (nanoflann.hpp:858-1004 build, :1278-1410 radius search): its search kernels.  The
// build kernels are in k_index_build.cuh.
//
// Layout (see IndexView in sb_device.cuh): the N-5 window points value[w..w+5]
// (sigmap_adaptor.h:89-97) are put into the aligned KD order (k_index_build.cuh) and cut into 8-point leaves;
// 8 consecutive leaves / nodes form the next level's node, pointer-free.  A query is handled by ONE WARP that advances EIGHT tree nodes (or
// eight leaves) per step, two per 8-lane group: every lane tests two child boxes (three 8-byte
// loads each) or evaluates two points, so each step keeps six independent loads per lane in
// flight and the whole warp stays busy at fan-out 8 -- where a 6-D hierarchy prunes far better
// than at fan-out 32 (the ball of radius 0.28 meets ~30 8-point leaves but ~28 32-point blocks:
// 4x fewer points to evaluate, 2.5x fewer boxes to test).
//
// Exactness: the accept test is the reference's own fp32 expression
//   d2 = ((e0+e1)+e2)+e3, then +e4, +e5, e_k = (q_k - v_k)^2, accept iff d2 < radius
// (nanoflann.hpp:383-408, :249-251, :1362; the "radius" is already squared, Q4) without FMA.
// Boxes only prune: their binary16 corners are rounded outwards when built and the tests keep a
// slack on the squared radius (box_d2_h; 1e-4 relative in the general kernel), so no point the
// exact test would accept is ever lost.
#ifndef SB_K_INDEX_CUH
#define SB_K_INDEX_CUH

#include <cuda_fp16.h>

#include "sb_device.cuh"

namespace sb {

// ------------------------------------------------------------------ search
//
// Two kernels share the work of radiusSearch (spatial_index.cc:366):
//
//   k_search_lean     the fast path, one 1024-thread CTA per SM.  Queries arrive sorted by the
//                     Morton code of the query point (k_query_keys + a radix sort), so the warps
//                     in flight walk the same corner of the index and nodes / leaves come from
//                     L1/L2 instead of DRAM.  The node levels every query walks (the prefix of
//                     nodes[] that fits 64 KB) are staged in shared memory with one TMA bulk copy
//                     (cp.async.bulk + mbarrier).  A warp owns a query and walks the hierarchy
//                     level by level: the frontier of one level sits in shared memory, every step
//                     tests the 64 child boxes of eight frontier nodes (two per 8-lane group, packed
//                     binary16 arithmetic) and appends the survivors to the next level's frontier;
//                     the last frontier holds leaves, evaluated the same way with the exact fp32
//                     expression.  No stacks, no per-level bookkeeping.  A query whose frontier would
//                     outgrow its kFrontCap slots is handed, untouched, to
//   k_radius_search   the general kernel (one small stack per level, any frontier size, the 5 000-hit
//                     cap of spatial_index.cc:371-372), which works through the list of such queries.
//                     A frontier of kFrontCap leaves holds 3 072 points, so a query that can reach the
//                     cap always takes this path: the cap rule lives in one place.
constexpr int kSearchWarps = 8;          // warps per CTA (general kernel)
constexpr int kLevelCap = 128;           // entries per level stack: 64 waiting + the children of one 8-node step
constexpr int kLeafQueueCap = 128;       // < 8 left over + 64 pushed per step
constexpr int kStageCap = 128;           // staged hits per warp before one global reservation
constexpr int kSearchGrab = 8;           // queries per grab of the dynamic work counter
constexpr int kMaxParts = 32;            // parts per entry the flush can route to (k_part_sort)
constexpr int kLeanWarps = 32;           // lean kernel: one 1024-thread CTA per SM
constexpr int kFrontCap = 384;           // lean kernel: frontier slots (nodes of a level / leaves) per query
constexpr int kLeanStage = 128;          // lean kernel: staged hits per warp, at least (SearchArgs::stage_cap: up to 256
                                         // where the staged top levels leave room, so that a query of a dense
                                         // index leaves one run per part instead of two or three short ones)
constexpr int kLeanStageMax = 256;       // ranks inside a part are 8 bits
constexpr int kLeanGrab = 4;             // lean kernel: sorted queries per grab
constexpr int kQueryBits = 12;           // query payload = entry << kQueryBits | query number inside the entry

// dynamic shared memory per warp of the general kernel: staging (key part, point id, d2), leaf
// queue, level counts, and one stack per node level
__host__ __device__ inline size_t search_smem_per_warp(int n_levels) {
  return (size_t)kStageCap * 16 + (size_t)kLeafQueueCap * 4 + 16 * 4 + kMaxParts * 4 +
         (size_t)n_levels * kLevelCap * 4;
}
// lean kernel, per warp: staged keys (8 B), distances and part|rank (2 B), two frontiers, per-part counts
__host__ __device__ inline size_t lean_warp_smem(uint32_t stage_cap) {
  return (size_t)stage_cap * 14 + 2 * (size_t)kFrontCap * 4 + kMaxParts * 4;
}
constexpr size_t kLeanWarpSmem = (size_t)kLeanStage * 14 + 2 * (size_t)kFrontCap * 4 + kMaxParts * 4;
constexpr size_t kLeanSmemLimit = 232448 - 1024;  // 227 KB per SM less the kernel's static shared memory
__host__ __device__ inline size_t lean_top_region(uint32_t smem_bytes) { return ((size_t)smem_bytes + 127) & ~(size_t)127; }
static_assert((size_t)kFrontCap * kLeaf < SMB_MAX_HITS, "the lean kernel must never be able to reach the hit cap");
static_assert(kLeanStage >= 64 && kLeanStageMax <= 256, "a leaf step stages up to 64 hits; ranks are 8 bits");
__host__ __device__ inline size_t lean_smem(uint32_t smem_bytes, uint32_t stage_cap) {
  return lean_top_region(smem_bytes) + (size_t)kLeanWarps * lean_warp_smem(stage_cap);
}
// the largest staging size (a multiple of 32) that fits next to the staged top levels
__host__ inline uint32_t lean_stage_cap(uint32_t smem_bytes) {
  uint32_t s = (uint32_t)kLeanStageMax;
  while (s > (uint32_t)kLeanStage && lean_smem(smem_bytes, s) > kLeanSmemLimit) s -= 32u;
  return s;
}

struct SearchArgs {
  // queries: either pipeline mode (features of batch entries) or stage mode (explicit)
  const float *features;       // pipeline: rows of kFeatCap floats; stage: [nq][6]
  const uint32_t *feat_row;    // pipeline: feature row of each batch entry
  const uint32_t *q_off;       // pipeline: exclusive scan of queries per entry, B+1 entries
  const uint32_t *entry_slot;  // pipeline: batch entry -> slot
  const SlotState *slots;      // pipeline: num_events (query offset) per slot
  uint32_t B;
  uint32_t n_queries;          // stage mode; pipeline reads q_off[B]
  int step;
  float radius;                // squared L2 (Q4)
  KeyLayout key;
  uint64_t *out_key;
  float *out_dist;
  unsigned long long cap;      // capacity of out_key/out_dist
  Counters *ctr;
  SlotState *slots_mut;        // to flag capped queries
  // pipeline mode: where each entry's hits went (k_sort.cuh); runs == nullptr disables it.
  // Every flush routes its hits to the n_parts coordinate ranges ("parts": part_of(g) with
  // g = bucket_base[bucket] + target) of the entry and records one run per part it touched.
  RunRec *runs;                // [B * n_parts][runs_cap]
  uint32_t *run_count;         // [B * n_parts]
  uint32_t *entry_total;       // [B * n_parts] anchors per (entry, part) so far
  uint32_t runs_cap;
  uint32_t n_parts;            // 1..kMaxParts
  float inv_span;              // 1 / coordinates per part
  const uint64_t *bucket_base;
  uint32_t n_buckets;
  unsigned int *work;          // the work counter of this launch
  // lean kernel: queries in Morton order.  order[k] = payload of the k-th query (pipeline:
  // entry << kQueryBits | query number; stage: query id); nullptr = natural order.
  const uint32_t *order;
  uint32_t nq_cap;             // pipeline: capacity of order[] (sized from an estimate; more queries
                               // than that raise error bit 6 and the host redoes the step)
  const uint2 *entry_info;     // pipeline: {feature row, query offset (num_events)} per entry
  uint32_t front_cap;          // frontier slots a query may use (<= kFrontCap; tests lower it)
  uint32_t stage_cap;          // lean kernel: staged hits per warp (kLeanStage .. kLeanStageMax, multiple of 32)
  uint32_t *ovf_list;          // payloads of the queries left to the general kernel
  // general kernel: qlist != nullptr -> work through qlist[0 .. *qlist_n) instead of all queries
  const uint32_t *qlist;
  const unsigned int *qlist_n;
};

__device__ __forceinline__ float exact_d2(const float q[kDim], const float v[kDim]) {
  float e[kDim];
#pragma unroll
  for (int d = 0; d < kDim; ++d) {
    float t = __fsub_rn(q[d], v[d]);
    e[d] = __fmul_rn(t, t);
  }
  float r = __fadd_rn(__fadd_rn(__fadd_rn(e[0], e[1]), e[2]), e[3]);
  r = __fadd_rn(r, e[4]);
  r = __fadd_rn(r, e[5]);
  return r;
}

// largest entry e in [0, B) with q_off[e] <= qi (q_off is non-decreasing, q_off[0] = 0 <= qi
// < q_off[B]); 32-ary search by the whole warp: three rounds for 32 K entries
__device__ __forceinline__ uint32_t find_entry(const uint32_t *__restrict__ q_off, uint32_t B, uint32_t qi,
                                               int lane) {
  uint32_t lo = 0, hi = B;
  while (hi - lo > 1) {
    const uint32_t stride = (hi - lo + 31u) / 32u;
    const uint32_t idx = lo + stride * (uint32_t)lane;
    const bool le = idx < hi && __ldg(q_off + idx) <= qi;
    const int k = __popc(__ballot_sync(0xffffffffu, le)) - 1;  // lane 0 (idx = lo) is always true
    lo += stride * (uint32_t)k;
    hi = min(lo + stride, hi);
  }
  return lo;
}

// ---- Morton order of the queries (lean kernel).  One block per batch entry; key = 24-bit Morton
// code (6 dims x 4 bits) of the query point in the index's own quantisation, payload =
// entry << kQueryBits | query number.  Also fills entry_info.
__device__ __forceinline__ uint32_t morton24(const float *q, float vmin, float inv_span) {
  uint32_t c = 0;
#pragma unroll
  for (int d = 0; d < kDim; ++d) {
    int v = (int)((q[d] - vmin) * inv_span * 16.0f);
    v = v < 0 ? 0 : (v > 15 ? 15 : v);
#pragma unroll
    for (int b = 0; b < 4; ++b) c |= (uint32_t)((v >> b) & 1) << (kDim * b + (kDim - 1 - d));
  }
  return c;
}

__global__ void k_query_keys(const float *__restrict__ features, const uint32_t *__restrict__ feat_row,
                             const uint32_t *__restrict__ q_off, const uint32_t *__restrict__ entry_slot,
                             const SlotState *__restrict__ slots, uint32_t B, int step, float vmin,
                             float inv_span, uint32_t *__restrict__ key, uint32_t *__restrict__ payload,
                             uint2 *__restrict__ entry_info, uint32_t nq_cap) {
  const uint32_t b = blockIdx.x;
  if (b >= B) return;
  const uint32_t q0 = q_off[b], nq = q_off[b + 1] - q0;
  const uint32_t frow = feat_row[b];
  if (threadIdx.x == 0) entry_info[b] = make_uint2(frow, slots[entry_slot[b]].num_events);
  const float *f = features + (size_t)frow * kFeatCap;
  for (uint32_t k = threadIdx.x; k < nq && q0 + k < nq_cap; k += blockDim.x) {
    const uint32_t p = (uint32_t)step * (k + 1u);  // seeds at step, 2*step, ... (Q3)
    float q[kDim];
#pragma unroll
    for (int d = 0; d < kDim; ++d) q[d] = f[p + d];
    key[q0 + k] = morton24(q, vmin, inv_span);
    payload[q0 + k] = (b << kQueryBits) | k;
  }
}

// natural query order (small batches): only the per-entry table
__global__ void k_entry_info(const uint32_t *__restrict__ feat_row, const uint32_t *__restrict__ entry_slot,
                             const SlotState *__restrict__ slots, uint32_t B, uint2 *__restrict__ entry_info) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) entry_info[b] = make_uint2(feat_row[b], slots[entry_slot[b]].num_events);
}

// stage mode: Morton keys of explicit queries, payload = query id
__global__ void k_query_keys_stage(const float *__restrict__ queries, uint32_t nq, float vmin, float inv_span,
                                   uint32_t *__restrict__ key, uint32_t *__restrict__ payload) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  float q[kDim];
#pragma unroll
  for (int d = 0; d < kDim; ++d) q[d] = queries[(size_t)i * kDim + d];
  key[i] = morton24(q, vmin, inv_span);
  payload[i] = i;
}

// ---- hits -> global memory.  `n` staged (key, d2) pairs of ONE batch entry: one reservation of
// output space, the hits grouped by coordinate part inside it, one run record per part touched.
// Not inlined: it is called from three places of two kernels and is off the traversal's path.
__device__ __noinline__ void flush_routed(const SearchArgs &a, const uint64_t *__restrict__ st_key,
                                          const float *__restrict__ st_dist, uint16_t *__restrict__ st_where,
                                          uint32_t *__restrict__ pcnt, const uint64_t *__restrict__ s_bb, int n,
                                          uint32_t entry) {
  const int lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  pcnt[lane] = 0;
  __syncwarp();
  // pass 1: part of every hit and its rank inside the part (part << 8 | rank, kept in shared memory)
  for (int i = lane; i < n; i += 32) {
    const uint64_t key = st_key[i];
    const uint32_t b = a.key.bucket(key);
    const uint64_t base = s_bb ? s_bb[b] : __ldg(a.bucket_base + b);
    const uint32_t part = part_of(base + a.key.target(key), a.inv_span, a.n_parts);
    st_where[i] = (uint16_t)((part << 8) | atomicAdd(&pcnt[part], 1u));
  }
  __syncwarp();
  const uint32_t mine = pcnt[lane];  // lane p: hits of part p
  uint32_t incl = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(full, incl, d);
    if (lane >= d) incl += t;
  }
  const uint32_t excl = incl - mine;
  // both reservations are issued before either result is used: one round trip, not two
  const size_t list = (size_t)entry * a.n_parts + lane;
  uint32_t r = 0;
  if (mine) r = atomicAdd(&a.run_count[list], 1u);
  unsigned long long base = 0;
  if (lane == 0) base = atomicAdd(&a.ctr->n_anchors, (unsigned long long)n);
  base = __shfl_sync(full, base, 0);
  if (mine) {
    if (r < a.runs_cap) a.runs[list * a.runs_cap + r] = RunRec{(uint32_t)(base + excl), mine};
    else atomicOr(&a.ctr->error, 8u);
    atomicAdd(&a.entry_total[list], mine);
  }
  pcnt[lane] = excl;  // offset of part p inside this flush
  __syncwarp();
  // pass 2: every hit to its place
  for (int i = lane; i < n; i += 32) {
    const uint32_t wh = st_where[i];
    const unsigned long long o = base + pcnt[wh >> 8] + (wh & 0xFFu);
    if (o < a.cap) {
      a.out_key[o] = st_key[i];
      a.out_dist[o] = st_dist[i];
    }
  }
  __syncwarp();
}

// the same without routing (stage mode; pipeline mode on the radix-sort path)
template <int CAP>
__device__ __noinline__ void flush_plain(const SearchArgs &a, const uint64_t *__restrict__ st_key,
                                         const float *__restrict__ st_dist, int n) {
  const int lane = threadIdx.x & 31;
  unsigned long long base = 0;
  if (lane == 0) base = atomicAdd(&a.ctr->n_anchors, (unsigned long long)n);
  base = __shfl_sync(0xffffffffu, base, 0);
  for (int i = lane; i < n; i += 32) {  // n <= CAP
    const unsigned long long o = base + i;
    if (o < a.cap) {
      a.out_key[o] = st_key[i];
      a.out_dist[o] = st_dist[i];
    }
  }
  __syncwarp();
}

// ---- the packed binary16 box test.  It stays conservative through a per-query threshold: with
// qh = round16(q) (|qh - q| <= 2^-11 |q|) every per-dimension distance computed in binary16 is at
// most (T_d + 2^-11 |q_d|)(1 + 2^-11) where T_d is the exact distance to the stored box (itself
// rounded outwards), so a box within r of q gives a sum of squares of at most
// (r + 2^-11 |q|_2)^2 (1 + 2^-11)^8; anything above that is pruned.  Overflow gives +inf (pruned,
// correctly: such a box is farther than 65504 - |q|), inf - inf gives NaN, which max() drops.
struct QueryH {
  __half2 q01, q23, q45;
  float theta;
};
// r = sqrt(r2) is computed once per kernel; |q|_2 is bounded by sqrt(6) max|q_d| (no square root
// per query: the bound only has to be an upper one)
__device__ __forceinline__ QueryH make_query_h(const float q[kDim], float r) {
  QueryH h;
  h.q01 = __floats2half2_rn(q[0], q[1]);
  h.q23 = __floats2half2_rn(q[2], q[3]);
  h.q45 = __floats2half2_rn(q[4], q[5]);
  float qmax = 0.0f;
#pragma unroll
  for (int d = 0; d < kDim; ++d) qmax = fmaxf(qmax, fabsf(q[d]));
  const float reach = r + 4.8828125e-4f * 2.4495f * qmax * 1.001f;  // r + 2^-11 sqrt(6) max|q_d| >= r + 2^-11 |q|_2
  h.theta = reach * reach * 1.0045f + 1e-6f;                          // (1 + 2^-11)^8 < 1.004; + underflow slack
  return h;
}
__device__ __forceinline__ float box_d2_h(const uint2 r0, const uint2 r1, const uint2 r2, const QueryH &h) {
  auto as_h2 = [](uint32_t v) { return *reinterpret_cast<const __half2 *>(&v); };
  const __half2 zero = __float2half2_rn(0.0f);
  const __half2 t01 = __hmax2(__hmax2(__hsub2(as_h2(r0.x), h.q01), __hsub2(h.q01, as_h2(r1.y))), zero);
  const __half2 t23 = __hmax2(__hmax2(__hsub2(as_h2(r0.y), h.q23), __hsub2(h.q23, as_h2(r2.x))), zero);
  const __half2 t45 = __hmax2(__hmax2(__hsub2(as_h2(r1.x), h.q45), __hsub2(h.q45, as_h2(r2.y))), zero);
  __half2 acc = __hmul2(t01, t01);
  acc = __hfma2(t23, t23, acc);
  acc = __hfma2(t45, t45, acc);
  return __low2float(acc) + __high2float(acc);
}

// ---- TMA bulk copy global -> shared, completion on an mbarrier (sm_90+: UBLKCP)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// One level of the lean traversal: the nf frontier nodes in src[] -> the surviving children in
// dst[]; returns their number, or -1 when dst would outgrow front_cap.  SMEM: the level's records
// are in shared memory.  Eight nodes per step (two per 8-lane group: six independent loads per lane
// in flight), then the tail of at most four.  (Sixteen per step was measured: 18 % more warp
// instructions for the same time -- the extra registers cost more than the shared loop overhead.)
template <bool SMEM>
__device__ __forceinline__ uint2 node_ld(const uint2 *p) {
  return SMEM ? *p : __ldg(p);
}
template <bool SMEM>
__device__ __forceinline__ int lean_node_level(const uint2 *__restrict__ lvl, const uint32_t *__restrict__ src,
                                               uint32_t *__restrict__ dst, int nf, int front_cap, const QueryH &qh,
                                               int lane, int grp, int sub, unsigned lt) {
  const unsigned full = 0xffffffffu;
  int nn = 0, i0 = 0;
  for (; i0 < nf; i0 += 8) {
    if (nn > front_cap - 64) return -1;
    const int ia = i0 + grp, ib = ia + 4;
    const bool hasA = ia < nf, hasB = ib < nf;
    const uint32_t nodeA = hasA ? src[ia] : 0u;
    const uint2 *ra = lvl + (size_t)nodeA * kNodeRec + sub;
    const uint2 a0 = node_ld<SMEM>(ra), a1 = node_ld<SMEM>(ra + kFan), a2 = node_ld<SMEM>(ra + 2 * kFan);
    if (i0 + 4 < nf) {  // a full step: two nodes per lane group
      const uint32_t nodeB = hasB ? src[ib] : 0u;
      const uint2 *rb = lvl + (size_t)nodeB * kNodeRec + sub;
      const uint2 b0 = node_ld<SMEM>(rb), b1 = node_ld<SMEM>(rb + kFan), b2 = node_ld<SMEM>(rb + 2 * kFan);
      const float sa = box_d2_h(a0, a1, a2, qh), sb = box_d2_h(b0, b1, b2, qh);
      const unsigned mA = __ballot_sync(full, hasA && sa <= qh.theta);
      const unsigned mB = __ballot_sync(full, hasB && sb <= qh.theta);
      const int nA = __popc(mA);
      if ((mA >> lane) & 1u) dst[nn + __popc(mA & lt)] = nodeA * kFan + sub;
      if ((mB >> lane) & 1u) dst[nn + nA + __popc(mB & lt)] = nodeB * kFan + sub;
      nn += nA + __popc(mB);
    } else {  // the level's tail: at most four nodes
      const float sa = box_d2_h(a0, a1, a2, qh);
      const unsigned mA = __ballot_sync(full, hasA && sa <= qh.theta);
      if ((mA >> lane) & 1u) dst[nn + __popc(mA & lt)] = nodeA * kFan + sub;
      nn += __popc(mA);
    }
  }
  __syncwarp();
  return nn;
}

// STAGE=false: hits become sort keys (entry|bucket|target|query) + d2 (never capped here: a
// frontier of kFrontCap = 384 leaves holds 3 072 points, fewer than the cap of 5 000).
// STAGE=true : key = query_id << 32 | window index (parity hook, compared as sets).
template <bool STAGE>
__global__ void __launch_bounds__(kLeanWarps * 32, 1)
k_search_lean(const __grid_constant__ IndexView ix, const __grid_constant__ SearchArgs a) {
  extern __shared__ __align__(128) unsigned char s_dyn[];
  __shared__ __align__(8) unsigned long long s_mbar;
  __shared__ uint64_t s_bb_store[64];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int grp = lane >> 3, sub = lane & 7;
  const unsigned full = 0xffffffffu;
  const unsigned lt = (1u << lane) - 1u;
  const uint2 *s_top = reinterpret_cast<const uint2 *>(s_dyn);
  const int stage_cap = (int)a.stage_cap;
  unsigned char *mine = s_dyn + lean_top_region(ix.smem_bytes) + (size_t)wid * lean_warp_smem(a.stage_cap);
  uint64_t *st_key = reinterpret_cast<uint64_t *>(mine);
  float *st_dist = reinterpret_cast<float *>(mine + (size_t)stage_cap * 8);
  uint32_t *fa = reinterpret_cast<uint32_t *>(mine + (size_t)stage_cap * 12);
  uint32_t *fb = fa + kFrontCap;
  uint32_t *pcnt = fb + kFrontCap;
  uint16_t *st_where = reinterpret_cast<uint16_t *>(pcnt + kMaxParts);

  // ---- the top levels: one bulk copy per CTA, everybody waits on the mbarrier
  if (threadIdx.x == 0) mbar_init(&s_mbar, 1);
  __syncthreads();
  if (threadIdx.x == 0 && ix.smem_bytes) {
    mbar_expect_tx(&s_mbar, ix.smem_bytes);
    bulk_g2s(s_dyn, ix.nodes, ix.smem_bytes, &s_mbar);
  }
  const bool bb_local = !STAGE && a.runs && a.n_buckets <= 64u;
  if (bb_local && threadIdx.x < a.n_buckets) s_bb_store[threadIdx.x] = a.bucket_base[threadIdx.x];
  const uint64_t *s_bb = bb_local ? s_bb_store : nullptr;
  __syncthreads();
  if (ix.smem_bytes) mbar_wait(&s_mbar, 0);

  uint32_t nq = STAGE ? a.n_queries : a.q_off[a.B];
  if (!STAGE && nq > a.nq_cap) {
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(&a.ctr->error, 64u);
    nq = a.nq_cap;
  }
  const float r2 = a.radius;
  const float r_up = sqrtf(r2) * 1.000001f;  // an upper bound of the radius itself
  const int top_level = ix.n_levels - 1;
  const int n_top = (int)ix.level_count[top_level];  // <= 8
  const int front_cap = (int)a.front_cap;
  const uint32_t grab = (uint32_t)kLeanGrab;
  const bool routed = !STAGE && a.runs;
  int staged = 0;
  uint32_t staged_entry = 0;
  unsigned long long my_hits = 0;
  uint32_t n_entry = 0, n_q0 = 1, n_q1 = 0;  // natural order: the entry of the previous query and its range

  for (;;) {
    uint32_t q0 = 0;
    if (lane == 0) q0 = atomicAdd(a.work, grab);
    q0 = __shfl_sync(full, q0, 0);
    if (q0 >= nq) break;
    const uint32_t q1 = min(q0 + grab, nq);
    for (uint32_t qi = q0; qi < q1; ++qi) {
      // ---- the query
      uint32_t payload = qi;  // stage mode: the query id
      if (a.order) {
        payload = __ldg(a.order + qi);
      } else if (!STAGE) {  // natural order: consecutive queries mostly share their entry
        if (qi < n_q0 || qi >= n_q1) {
          n_entry = find_entry(a.q_off, a.B, qi, lane);
          n_q0 = __ldg(a.q_off + n_entry);
          n_q1 = __ldg(a.q_off + n_entry + 1);
        }
        payload = (n_entry << kQueryBits) | (qi - n_q0);
      }
      float q[kDim];
      uint64_t qk;
      uint32_t entry = 0;
      if (STAGE) {
#pragma unroll
        for (int d = 0; d < kDim; ++d) q[d] = __ldg(a.features + (size_t)payload * kDim + d);
        qk = (uint64_t)payload << 32;
      } else {
        entry = payload >> kQueryBits;
        const uint2 info = __ldg(a.entry_info + entry);
        const uint32_t p = (uint32_t)a.step * ((payload & ((1u << kQueryBits) - 1u)) + 1u);
        const float *f = a.features + (size_t)info.x * kFeatCap + p;
#pragma unroll
        for (int d = 0; d < kDim; ++d) q[d] = __ldg(f + d);
        qk = a.key.pack(entry, 0u, 0u, p + info.y);
        if (routed && staged && entry != staged_entry) {
          flush_routed(a, st_key, st_dist, st_where, pcnt, s_bb, staged, staged_entry);
          staged = 0;
        }
        staged_entry = entry;
      }
      // a NaN coordinate (a chunk whose event means are all equal: 0/0 in the z-score) matches
      // nothing in the reference (nanoflann: NaN < radius is false) -- and would pass every box test here
      if (!(fabsf(q[0] + q[1] + q[2] + q[3] + q[4] + q[5]) <= 3.0e38f)) continue;
      const QueryH qh = make_query_h(q, r_up);

      // ---- node levels, top down
      int nf = n_top;
      if (lane < n_top) fa[lane] = (uint32_t)lane;
      __syncwarp();
      uint32_t *src = fa, *dst = fb;
      for (int L = top_level; L >= 0 && nf > 0; --L) {
        const uint32_t off = ix.level_off[L];
        if (L >= ix.smem_from) nf = lean_node_level<true>(s_top + off, src, dst, nf, front_cap, qh, lane, grp, sub, lt);
        else nf = lean_node_level<false>(ix.nodes + off, src, dst, nf, front_cap, qh, lane, grp, sub, lt);
        uint32_t *t = src;
        src = dst;
        dst = t;
      }
      if (nf < 0) {  // frontier too large: the general kernel takes this query from scratch
        if (lane == 0) a.ovf_list[atomicAdd(&a.ctr->n_overflow, 1u)] = payload;
        continue;
      }

      // ---- leaves: eight per step, one point per lane and half step
      for (int i0 = 0; i0 < nf; i0 += 8) {
        const int ia = i0 + grp, ib = ia + 4;
        const bool hasA = ia < nf, hasB = ib < nf;
        const uint32_t leafA = hasA ? src[ia] : 0u, leafB = hasB ? src[ib] : 0u;
        const uint2 *la = ix.leaves + (size_t)leafA * kLeafRec + sub;
        const uint2 *lb = ix.leaves + (size_t)leafB * kLeafRec + sub;
        const uint2 a01 = __ldg(la), a23 = __ldg(la + kLeaf), a45 = __ldg(la + 2 * kLeaf);
        const uint2 b01 = __ldg(lb), b23 = __ldg(lb + kLeaf), b45 = __ldg(lb + 2 * kLeaf);
        const float va[kDim] = {__uint_as_float(a01.x), __uint_as_float(a01.y), __uint_as_float(a23.x),
                                __uint_as_float(a23.y), __uint_as_float(a45.x), __uint_as_float(a45.y)};
        const float vb[kDim] = {__uint_as_float(b01.x), __uint_as_float(b01.y), __uint_as_float(b23.x),
                                __uint_as_float(b23.y), __uint_as_float(b45.x), __uint_as_float(b45.y)};
        const float d2a = exact_d2(q, va), d2b = exact_d2(q, vb);
        const unsigned hitA = __ballot_sync(full, hasA && d2a < r2);
        const unsigned hitB = __ballot_sync(full, hasB && d2b < r2);
        if (hitA | hitB) {
          const int nA = __popc(hitA), nh = nA + __popc(hitB);
          if (staged + nh > stage_cap) {
            if (routed) flush_routed(a, st_key, st_dist, st_where, pcnt, s_bb, staged, staged_entry);
            else flush_plain<kLeanStageMax>(a, st_key, st_dist, staged);
            staged = 0;
          }
          if ((hitA >> lane) & 1u) {
            const int at = staged + __popc(hitA & lt);
            uint64_t key;
            if (STAGE) {
              key = qk | __ldg(ix.leaf_widx + (size_t)leafA * kLeaf + sub);
            } else {
              const uint2 tb = __ldg(la + 3 * kLeaf);
              key = qk | ((uint64_t)tb.y << a.key.sh_b()) | ((uint64_t)tb.x << a.key.sh_t());
            }
            st_key[at] = key;
            st_dist[at] = d2a;
          }
          if ((hitB >> lane) & 1u) {
            const int at = staged + nA + __popc(hitB & lt);
            uint64_t key;
            if (STAGE) {
              key = qk | __ldg(ix.leaf_widx + (size_t)leafB * kLeaf + sub);
            } else {
              const uint2 tb = __ldg(lb + 3 * kLeaf);
              key = qk | ((uint64_t)tb.y << a.key.sh_b()) | ((uint64_t)tb.x << a.key.sh_t());
            }
            st_key[at] = key;
            st_dist[at] = d2b;
          }
          __syncwarp();
          staged += nh;
          my_hits += (unsigned)nh;
        }
      }
      __syncwarp();  // frontier reads are done before the next query refills it
    }
  }
  if (staged) {
    if (routed) flush_routed(a, st_key, st_dist, st_where, pcnt, s_bb, staged, staged_entry);
    else flush_plain<kLeanStageMax>(a, st_key, st_dist, staged);
  }
  if (lane == 0 && my_hits) atomicAdd(&a.ctr->n_hits, my_hits);
}

// ---- the general kernel.
// STAGE=false: hits become sort keys (entry|bucket|target|query) + d2, capped at 5000/query.
// STAGE=true : key = query_id << 32 | window index, no cap (parity hook, compared as sets).
//
// Traversal: level-order over one small stack per level, eight nodes wide.  The warp works on the
// HIGHEST level with waiting nodes as long as the stack below has room for the 64 children of a
// step (else on the lowest one, whose child stack is empty), so every level is consumed in full
// groups of eight nodes with at most one partial group per level; it pops up to eight nodes (two
// per 8-lane group), tests their 64 child boxes with six independent loads per lane in flight,
// and pushes the survivors onto the stack of the level below.  Surviving leaves queue up and are
// evaluated eight at a time the same way.  Any frontier size works: a full stack just forces the
// walk down to the leaves before the level above is continued.
template <bool STAGE>
__global__ void __launch_bounds__(kSearchWarps * 32, 4)
k_radius_search(const __grid_constant__ IndexView ix, const __grid_constant__ SearchArgs a) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int grp = lane >> 3, sub = lane & 7;
  const unsigned full = 0xffffffffu;
  const unsigned lt = (1u << lane) - 1u;
  const int n_levels = ix.n_levels;
  unsigned char *mine = s_dyn + (size_t)wid * search_smem_per_warp(n_levels);
  uint64_t *st_key = reinterpret_cast<uint64_t *>(mine);
  float *st_dist = reinterpret_cast<float *>(mine + kStageCap * 8);
  uint16_t *st_where = reinterpret_cast<uint16_t *>(mine + kStageCap * 12);
  uint32_t *leafq = reinterpret_cast<uint32_t *>(mine + kStageCap * 16);
  uint32_t *lcnt = leafq + kLeafQueueCap;          // [16] nodes waiting per level
  uint32_t *pcnt = lcnt + 16;                      // [kMaxParts] hits per part of the flush in progress
  uint32_t *lstk = pcnt + kMaxParts;               // [n_levels][kLevelCap]
  const uint32_t nq = a.qlist ? *a.qlist_n : (STAGE ? a.n_queries : a.q_off[a.B]);
  const float r2 = a.radius;
  const float r2_prune = r2 * 1.0001f + 1e-12f;
  const uint32_t grab = a.qlist ? 1u : (uint32_t)kSearchGrab;
  const int top_level = n_levels - 1;
  const uint32_t n_top = ix.level_count[top_level];  // <= 8
  const bool routed = !STAGE && a.runs;
  int staged = 0;
  unsigned long long my_hits = 0, my_capped = 0;
  // entry of the previous query and its query range (consecutive queries mostly share it)
  uint32_t entry = 0, e_q0 = 1, e_q1 = 0, slot = 0, ev_off = 0, frow = 0;
  uint32_t staged_entry = 0;  // the entry every staged hit belongs to (a run never mixes entries)

  auto flush = [&]() {
    if (staged == 0) return;
    if (routed) flush_routed(a, st_key, st_dist, st_where, pcnt, nullptr, staged, staged_entry);
    else flush_plain<kStageCap>(a, st_key, st_dist, staged);
    staged = 0;
  };

  for (;;) {
    uint32_t q0 = 0;
    if (lane == 0) q0 = atomicAdd(a.work, grab);
    q0 = __shfl_sync(full, q0, 0);
    if (q0 >= nq) break;
    const uint32_t q1 = min(q0 + grab, nq);
    for (uint32_t qi = q0; qi < q1; ++qi) {
      // ---- locate the query
      float q[kDim];
      uint64_t qk;
      if (STAGE) {
        const uint32_t id = a.qlist ? __ldg(a.qlist + qi) : qi;
#pragma unroll
        for (int d = 0; d < kDim; ++d) q[d] = __ldg(a.features + (size_t)id * kDim + d);
        qk = (uint64_t)id << 32;
      } else {
        uint32_t p;
        if (a.qlist) {
          const uint32_t payload = __ldg(a.qlist + qi);
          const uint32_t e = payload >> kQueryBits;
          if (e != entry || e_q1 == 0) {
            flush();
            entry = e;
            e_q1 = 1;  // marks `entry` valid
            slot = __ldg(a.entry_slot + entry);
            ev_off = a.slots[slot].num_events;
            frow = __ldg(a.feat_row + entry);
          }
          staged_entry = entry;
          p = (uint32_t)a.step * ((payload & ((1u << kQueryBits) - 1u)) + 1u);
        } else {
          if (qi < e_q0 || qi >= e_q1) {
            flush();
            entry = find_entry(a.q_off, a.B, qi, lane);
            staged_entry = entry;
            e_q0 = __ldg(a.q_off + entry);
            e_q1 = __ldg(a.q_off + entry + 1);
            slot = __ldg(a.entry_slot + entry);
            ev_off = a.slots[slot].num_events;  // query_start_offset
            frow = __ldg(a.feat_row + entry);
          }
          p = (uint32_t)a.step * (qi - e_q0 + 1u);  // seeds at step, 2*step, ... (Q3)
        }
        const float *f = a.features + (size_t)frow * kFeatCap + p;
#pragma unroll
        for (int d = 0; d < kDim; ++d) q[d] = __ldg(f + d);
        qk = a.key.pack(entry, 0u, 0u, p + ev_off);
      }
      if (!(fabsf(q[0] + q[1] + q[2] + q[3] + q[4] + q[5]) <= 3.0e38f)) continue;  // NaN: no hits (see k_search_lean)
      uint32_t qhits = 0;
      bool capped = false;
      // L = level being worked on (n_levels when none), c = how many wait there
      int L = top_level, c = (int)n_top, nleaf = 0;
      uint32_t waiting = 1u << top_level;  // levels with nodes on their stack
      if (lane < 16) lcnt[lane] = (lane == top_level) ? n_top : 0u;
      if (lane < (int)n_top) lstk[top_level * kLevelCap + lane] = (uint32_t)lane;
      __syncwarp();
      for (;;) {
        if (nleaf < 8 && waiting) {
          L = 31 - __clz(waiting);
          if (L > 0 && lcnt[L - 1] > (uint32_t)(kLevelCap - 64)) L = __ffs(waiting) - 1;
          c = (int)lcnt[L];
        } else {
          L = waiting ? 0 : n_levels;
        }
        if (nleaf >= 8 || (L >= n_levels && nleaf > 0)) {
          // ---- leaf step: up to eight leaves, two per 8-lane group, one point each per lane
          const int take = min(nleaf, 8);
          const bool hasA = grp < take, hasB = grp + 4 < take;
          const uint32_t leafA = hasA ? leafq[nleaf - 1 - grp] : 0u;
          const uint32_t leafB = hasB ? leafq[nleaf - 5 - grp] : 0u;
          nleaf -= take;
          const uint2 *la = ix.leaves + (size_t)leafA * kLeafRec + sub;
          const uint2 *lb = ix.leaves + (size_t)leafB * kLeafRec + sub;
          const uint2 a01 = __ldg(la), a23 = __ldg(la + kLeaf), a45 = __ldg(la + 2 * kLeaf);
          const uint2 b01 = __ldg(lb), b23 = __ldg(lb + kLeaf), b45 = __ldg(lb + 2 * kLeaf);
          const float va[kDim] = {__uint_as_float(a01.x), __uint_as_float(a01.y), __uint_as_float(a23.x),
                                  __uint_as_float(a23.y), __uint_as_float(a45.x), __uint_as_float(a45.y)};
          const float vb[kDim] = {__uint_as_float(b01.x), __uint_as_float(b01.y), __uint_as_float(b23.x),
                                  __uint_as_float(b23.y), __uint_as_float(b45.x), __uint_as_float(b45.y)};
          const float d2a = exact_d2(q, va), d2b = exact_d2(q, vb);
          const uint32_t hitA = __ballot_sync(full, hasA && d2a < r2);
          const uint32_t hitB = __ballot_sync(full, hasB && d2b < r2);
          __syncwarp();  // leafq reads are done before a later node step pushes
          bool stop = false;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            uint32_t hit = half ? hitB : hitA;
            if (!hit || stop) continue;
            if (!STAGE) {
              const uint32_t room = kMaxHits - qhits;
              if ((uint32_t)__popc(hit) > room) {
                // keep the first `room` hits in lane order (deterministic; see DESIGN.md H4)
                uint32_t keep = 0, m = hit;
                for (uint32_t k = 0; k < room; ++k) {
                  keep |= m & (0u - m);
                  m &= m - 1;
                }
                hit = keep;
                capped = true;
              }
            }
            const int nh = __popc(hit);
            if (staged + nh > kStageCap) flush();
            if (hit & (1u << lane)) {
              const int at = staged + __popc(hit & lt);
              const uint32_t leaf = half ? leafB : leafA;
              uint64_t key;
              if (STAGE) {
                key = qk | __ldg(ix.leaf_widx + (size_t)leaf * kLeaf + sub);
              } else {
                const uint2 tb = __ldg((half ? lb : la) + 3 * kLeaf);
                key = qk | ((uint64_t)tb.y << a.key.sh_b()) | ((uint64_t)tb.x << a.key.sh_t());
              }
              st_key[at] = key;
              st_dist[at] = half ? d2b : d2a;
            }
            __syncwarp();
            staged += nh;
            qhits += nh;
            if (!STAGE && qhits >= kMaxHits) {
              capped = true;  // conservatively: there may have been more than 5000
              stop = true;    // the reference stops taking hits after 5000 (spatial_index.cc:371-372)
            }
          }
          if (stop) break;
        } else if (L < n_levels) {
          // ---- node step: up to eight nodes of level L, two per 8-lane group
          const int take = min(c, 8);
          const bool hasA = grp < take, hasB = grp + 4 < take;
          const uint32_t *stk = lstk + L * kLevelCap;
          const uint32_t nodeA = hasA ? stk[c - 1 - grp] : 0u;
          const uint32_t nodeB = hasB ? stk[c - 5 - grp] : 0u;
          c -= take;
          const uint2 *base = ix.nodes + ix.level_off[L] + sub;
          const uint2 *ra = base + (size_t)nodeA * kNodeRec;
          const uint2 *rb = base + (size_t)nodeB * kNodeRec;
          const uint2 a0 = __ldg(ra), a1 = __ldg(ra + kFan), a2 = __ldg(ra + 2 * kFan);
          const uint2 b0 = __ldg(rb), b1 = __ldg(rb + kFan), b2 = __ldg(rb + 2 * kFan);
          // boxes only prune (stored rounded outwards, tested with slack), so this distance may
          // use FMA; the accept test may not
          float sa = 0.0f, sb = 0.0f;
          {
            const float2 l01 = unpack_h2(a0.x), l23 = unpack_h2(a0.y), l45 = unpack_h2(a1.x);
            const float2 h01 = unpack_h2(a1.y), h23 = unpack_h2(a2.x), h45 = unpack_h2(a2.y);
            const float lo[kDim] = {l01.x, l01.y, l23.x, l23.y, l45.x, l45.y};
            const float hi[kDim] = {h01.x, h01.y, h23.x, h23.y, h45.x, h45.y};
#pragma unroll
            for (int d = 0; d < kDim; ++d) {
              const float t = fmaxf(fmaxf(lo[d] - q[d], q[d] - hi[d]), 0.0f);
              sa = __fmaf_rn(t, t, sa);
            }
          }
          {
            const float2 l01 = unpack_h2(b0.x), l23 = unpack_h2(b0.y), l45 = unpack_h2(b1.x);
            const float2 h01 = unpack_h2(b1.y), h23 = unpack_h2(b2.x), h45 = unpack_h2(b2.y);
            const float lo[kDim] = {l01.x, l01.y, l23.x, l23.y, l45.x, l45.y};
            const float hi[kDim] = {h01.x, h01.y, h23.x, h23.y, h45.x, h45.y};
#pragma unroll
            for (int d = 0; d < kDim; ++d) {
              const float t = fmaxf(fmaxf(lo[d] - q[d], q[d] - hi[d]), 0.0f);
              sb = __fmaf_rn(t, t, sb);
            }
          }
          const uint32_t mA = __ballot_sync(full, hasA && sa <= r2_prune);
          const uint32_t mB = __ballot_sync(full, hasB && sb <= r2_prune);
          const int nA = __popc(mA), nB = __popc(mB);
          if (L > 0) {
            const uint32_t below = lcnt[L - 1];
            uint32_t *dst = lstk + (L - 1) * kLevelCap + below;
            if (mA & (1u << lane)) dst[__popc(mA & lt)] = nodeA * kFan + sub;
            if (mB & (1u << lane)) dst[nA + __popc(mB & lt)] = nodeB * kFan + sub;
            __syncwarp();  // every lane has read lcnt before lane 0 rewrites it
            if (lane == 0) {
              lcnt[L] = (uint32_t)c;
              lcnt[L - 1] = below + (uint32_t)(nA + nB);
            }
            if (nA + nB) waiting |= 1u << (L - 1);
          } else {
            if (mA & (1u << lane)) leafq[nleaf + __popc(mA & lt)] = nodeA * kFan + sub;
            if (mB & (1u << lane)) leafq[nleaf + nA + __popc(mB & lt)] = nodeB * kFan + sub;
            nleaf += nA + nB;
            __syncwarp();
            if (lane == 0) lcnt[0] = (uint32_t)c;
          }
          if (c == 0) waiting &= ~(1u << L);
          __syncwarp();
        } else {
          break;
        }
      }
      my_hits += qhits;
      if (capped) {
        ++my_capped;
        if (!STAGE && lane == 0) atomicOr(&a.slots_mut[slot].flags, 1u);
      }
    }
  }
  flush();
  if (lane == 0) {
    if (my_hits) atomicAdd(&a.ctr->n_hits, my_hits);
    if (my_capped) atomicAdd(&a.ctr->n_capped, my_capped);
  }
}

}  // namespace sb
#endif
