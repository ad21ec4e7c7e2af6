// k_chain.cuh -- K5..K7: anchors -> chains -> per-read decision, for a batch of read chunks.
//
// Input: the step's anchors as (64-bit key, d2) pairs already sorted by key =
// entry | bucket(contig*2+strand) | target | query, which is the reference's per-bucket
// std::sort order (spatial_index.cc:411-417, key spatial_index.h:22-25; (target, query) pairs
// are unique so the d2 tie-break never fires) with buckets in the reference's DP order
// (contig-major, '+' before '-', spatial_index.cc:420-422).
//
//   k_inject_carry   anchors of the previous chunk's surviving chains re-enter the buckets
//                    (spatial_index.cc:303-322), before the search appends its hits
//   k_fix_ties       (radix-sort path only) equal-target runs ordered by query
//   k_chain_prep     thread per anchor: coefficient, initial score, segment bounds and the
//                    position-only link test; linked anchors compacted into per-tile work lists
//   k_chain_dp       the banded chaining DP (spatial_index.cc:434-540), one WARP per
//                    (entry, bucket) segment over the linked anchors only -- buckets are
//                    independent until the running global max is applied
//   k_sel_trace      warp per segment: running max of the earlier buckets, traceback of the
//                    segment's <= 3 end candidates with used-flags (spatial_index.cc:165-220)
//   k_sel_scatter    contig-sharded runs: candidates gathered from the other ranks
//   k_sel_pick       warp per entry: primary chains (spatial_index.cc:222-253) and the carry-pool
//                    space they need; k_pool_check aborts the step if the pools are too small
//   k_sel_commit     warp per entry: MAPQ (spatial_index.cc:255-274), then StreamingMap's stop /
//                    output decision and tag sums (sigmap.cc:667-745); survivors' anchors go to
//                    the carry pool for the next chunk.
// All float arithmetic mirrors the reference expression by expression (no FMA).
#ifndef SB_K_CHAIN_CUH
#define SB_K_CHAIN_CUH

#include "sb_device.cuh"

namespace sb {

// per (entry, bucket) segment: where it lies in the sorted anchor array and what the DP
// found there.  Slot index = KeyLayout::seg(key) = entry << bbits | bucket, so the table is
// ordered like the reference's bucket loop by construction (no atomics, no scan).
struct SegRec {
  uint32_t start;     // first anchor of the segment; kSegEmpty = no anchors
  uint32_t end;       // one past the last anchor
  uint32_t ntop;      // local end candidates kept (<= 3)
  float max;          // max chaining score over the segment's linked anchors (see k_chain_dp)
  float top_s[3];     // best three local end candidates: score desc, index desc
  uint32_t top_i[3];
};
constexpr uint32_t kSegEmpty = 0xFFFFFFFFu;
constexpr int kPrepTile = 1024;  // anchors per k_chain_prep block = per compacted work list tile

struct ChainArgs {
  const uint64_t *key;   // sorted
  const float *dist;     // sorted alongside
  unsigned long long n_max;  // capacity of the anchor arrays; the count itself is ctr->n_anchors
  KeyLayout kl;
  float radius;
  float *score;
  float *coef;           // distance coefficient per anchor (k_chain_prep)
  uint32_t *pred;        // bit31 = anchor_is_used
  SegRec *seg;           // [n_slots], memset to 0xFF before k_chain_prep
  float *seg_max;        // [n_slots], zeroed: SegRec::max of every segment (0 when empty)
  uint32_t n_slots;      // B << bbits
  const uint32_t *seg_qmin;  // [n_slots] lower bound of the query positions in the segment (k_seg_qmin_init, k_inject_carry)
  uint32_t *link_list;   // [n_tiles * kPrepTile] indices of linked anchors, ascending per tile
  uint32_t *link_count;  // [n_tiles]
  uint16_t *pend_list;   // [n_tiles * kPrepTile] of those, the ones k_chain_prep could not settle itself
  uint32_t *pend_count;  //   (index inside the tile, ascending); [n_tiles]
  Counters *ctr;
  int dp_passes;         // thread-parallel passes of k_chain_dp before the in-order cooperative path
  int prep_rounds;       // settle rounds inside k_chain_prep (0: every linked anchor is left to the DP kernels)
};

// Every query of this step's chunk of an entry lies above the entry's event offset; carried anchors
// (older chunks) lower the bound of their own segment in k_inject_carry.  k_chain_prep's link test
// stops where no predecessor can be gap-compatible any more: 0.75 < dq/dt needs 3 dt < 4 dq, and
// dq <= q_i - seg_qmin.
__global__ void k_seg_qmin_init(const uint32_t *__restrict__ entry_slot, const SlotState *__restrict__ slots,
                                uint32_t n_slots, int bbits, uint32_t *__restrict__ seg_qmin) {
  const uint32_t sg = blockIdx.x * blockDim.x + threadIdx.x;
  if (sg < n_slots) seg_qmin[sg] = slots[entry_slot[sg >> bbits]].num_events;
}

constexpr int kCarryThreads = 256;
constexpr int kCarryMaxParts = 32;  // = kMaxParts of k_index.cuh

// runs == nullptr: no run lists (radix-sort path).  Otherwise the carried anchors of an entry are
// routed, 32 at a time, to the entry's n_parts coordinate ranges exactly like the hits of a search
// flush (k_index.cuh): one run per part touched.
__global__ void __launch_bounds__(kCarryThreads)
k_inject_carry(const uint32_t *__restrict__ entry_slot, const uint32_t *__restrict__ n_queries,
               const SlotState *__restrict__ slots, const CarryAnchor *__restrict__ pool0,
               const CarryAnchor *__restrict__ pool1, uint32_t B, KeyLayout kl,
               uint64_t *__restrict__ out_key, float *__restrict__ out_dist,
               unsigned long long cap, Counters *__restrict__ ctr, RunRec *__restrict__ runs,
               uint32_t *__restrict__ run_count, uint32_t *__restrict__ entry_total,
               uint32_t runs_cap, uint32_t n_parts, float inv_span, const uint64_t *__restrict__ bucket_base,
               uint32_t *__restrict__ seg_qmin) {
  __shared__ uint32_t s_cnt[kCarryThreads / 32][kCarryMaxParts];
  const uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) / 32, lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  if (b >= B) return;
  if (n_queries[b] == 0) return;  // GenerateChains is not called for this entry
  const SlotState st = slots[entry_slot[b]];
  if (st.carry_n == 0) return;
  const CarryAnchor *src = (st.pool ? pool1 : pool0) + st.carry_off;
  if (!runs) {
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(&ctr->n_anchors, (unsigned long long)st.carry_n);
    base = __shfl_sync(full, base, 0);
    for (uint32_t i = lane; i < st.carry_n; i += 32) {
      const CarryAnchor c = src[i];
      atomicMin(&seg_qmin[(b << kl.bbits) | c.bucket], c.query);
      if (base + i < cap) {
        out_key[base + i] = kl.pack(b, c.bucket, c.target, c.query);
        out_dist[base + i] = c.dist;
      }
    }
    return;
  }
  uint32_t *pcnt = s_cnt[(threadIdx.x >> 5)];
  for (uint32_t i0 = 0; i0 < st.carry_n; i0 += 32) {
    const uint32_t i = i0 + lane;
    const bool valid = i < st.carry_n;
    const uint32_t batch = min(32u, st.carry_n - i0);
    pcnt[lane] = 0;
    __syncwarp();
    CarryAnchor c = CarryAnchor{0u, 0u, 0.0f, 0u};
    uint32_t part = 0, rank = 0;
    if (valid) {
      c = src[i];
      atomicMin(&seg_qmin[(b << kl.bbits) | c.bucket], c.query);
      part = part_of(bucket_base[c.bucket] + c.target, inv_span, n_parts);
      rank = atomicAdd(&pcnt[part], 1u);
    }
    __syncwarp();
    const uint32_t mine = pcnt[lane];
    uint32_t incl = mine;
#pragma unroll
    for (int d = 1; d < kCarryMaxParts; d <<= 1) {
      const uint32_t t = __shfl_up_sync(full, incl, d);
      if (lane >= (uint32_t)d) incl += t;
    }
    const uint32_t excl = incl - mine;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(&ctr->n_anchors, (unsigned long long)batch);
    base = __shfl_sync(full, base, 0);
    if (mine) {
      const size_t list = (size_t)b * n_parts + lane;
      const uint32_t r = atomicAdd(&run_count[list], 1u);
      if (r < runs_cap) runs[list * runs_cap + r] = RunRec{(uint32_t)(base + excl), mine};
      else atomicOr(&ctr->error, 8u);
      atomicAdd(&entry_total[list], mine);
    }
    const uint32_t off = __shfl_sync(full, excl, (int)part);
    if (valid) {
      const unsigned long long o = base + off + rank;
      if (o < cap) {
        out_key[o] = kl.pack(b, c.bucket, c.target, c.query);
        out_dist[o] = c.dist;
      }
    }
    __syncwarp();
  }
}

// The radix sort skips the query bits (two passes fewer): it orders by (entry, bucket, target)
// and, being stable, leaves the rare anchors that share all three in arrival order.  This
// kernel finishes the reference's (target, query) order (spatial_index.h:22-25) by sorting
// each such run in place; (target, query) pairs are unique inside a segment, so the result
// is fully determined.  One thread per run head.
__global__ void k_fix_ties(uint64_t *__restrict__ key, float *__restrict__ dist, const Counters *__restrict__ ctr,
                           int lo_bits) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t n = (uint32_t)ctr->n_anchors;
  if (i >= n || ctr->abort) return;
  const uint64_t hi = key[i] >> lo_bits;
  if (i > 0 && (key[i - 1] >> lo_bits) == hi) return;  // inside a run: its head handles it
  uint32_t e = i + 1;
  while (e < n && (key[e] >> lo_bits) == hi) ++e;
  for (uint32_t x = i + 1; x < e; ++x) {  // insertion sort of [i, e) by the full key
    const uint64_t kk = key[x];
    const float dd = dist[x];
    uint32_t y = x;
    while (y > i && key[y - 1] > kk) {
      key[y] = key[y - 1];
      dist[y] = dist[y - 1];
      --y;
    }
    key[y] = kk;
    dist[y] = dd;
  }
}

constexpr int kBand = 5000;        // chaining_band_length, spatial_index.cc:286
constexpr int kMaxTargetGap = 5000;
constexpr int kMaxGap = 2000;
constexpr int kMaxSkips = 25;

// The chaining DP (spatial_index.cc:434-540) in two kernels.
//
// Anchors of one (entry, bucket) segment look strictly sequential: anchor i reads the scores
// of its predecessors.  But a predecessor j only ever changes anchor i's score if the pair
// passes the gap test (|dt - dq| < 2000 and 0.75 < dq/dt < 5, :499-520) inside the lookback
// range (same segment, i - j <= 5000, t_i - t_j <= 5000) -- and that test needs positions
// only, no scores.  At the reference's anchor density 80-88 % of the anchors (random
// background hits) have NO such predecessor: their score is the initial 6 * coef and their
// predecessor is themselves whatever the lookback does.  So:
//
//   k_chain_prep  one thread per anchor, fully parallel: initial score, pred = self, segment
//                 bounds, and the position-only test "is there any gap-compatible predecessor
//                 in the maximal lookback range" (a superset of the range the reference's
//                 skip counter actually visits).  Linked anchors are compacted, in order,
//                 into a per-tile work list.
//   k_chain_dp    one thread per segment walks only the linked anchors (5-8x fewer sequential
//                 steps) and runs the reference's lookback on them exactly: continue / break
//                 rules, running best, +-1 skip counter with its > 25 break.
//
// gap_scale tests as integers: 0.75 < fl(dq/dt) < 5  <=>  3*dt < 4*dq and dq < 5*dt, exact
// because dq/dt differs from either bound by >= 1/(4*dt) >= 5e-5 while fp32 rounding moves
// it by < 3e-7 (dt <= 5000 here, |dq| < 2^24).
__device__ __forceinline__ bool gap_compatible(int32_t dt, int32_t dq) {
  return abs(dt - dq) < kMaxGap && dq < 5 * dt && 4 * dq > 3 * dt;
}

// spatial_index.cc:438-444: 1 - 0.2 * distance / search_radius in double, then float
__device__ __forceinline__ float distance_coefficient(float dist, double radius) {
  return (float)__dsub_rn(1.0, __ddiv_rn(__dmul_rn(0.2, (double)dist), radius));
}

constexpr int kPrepHalo = 128;     // predecessors staged in shared memory ahead of the tile
constexpr int kPrepThreads = 256;  // kPrepTile / kPrepThreads anchors per thread
constexpr uint32_t kPending = 0x40000000u;  // pred[] bit: linked anchor not yet settled by the DP
constexpr int kPrepRounds = 1;     // settle rounds inside k_chain_prep

// Phase 2 of k_chain_prep: the lookback itself for the linked anchors it can finish on its own.
// 80-90 % of the linked anchors are background pairs and triples: their gap-compatible predecessors
// are unlinked anchors (score final = 6 * coef) a few places back, all inside the tile that is
// already unpacked in shared memory.  The tile's linked anchors, compacted, are taken one per
// thread; a thread runs the reference's lookback (continue/break rules, running best, +-1 skip
// counter with its > 25 break) over shared memory and settles its anchor iff every gap-compatible
// predecessor it meets is final -- unlinked, or settled in an EARLIER round (rounds are separated
// by barriers, so what a thread reads never depends on timing).  A predecessor in the halo (state
// unknown), a pending one, or a walk that runs off the staged range defers the anchor: it stays
// pending and goes to the tile's pending list for k_chain_dp, which then only walks the true-locus
// chains.
__global__ void __launch_bounds__(kPrepThreads, 8) k_chain_prep(ChainArgs a) {
  // the tile's anchors and the kPrepHalo before it, unpacked: {segment id, target, query, score bits}
  __shared__ int4 s_a[kPrepHalo + kPrepTile];
  constexpr int kSubTiles = kPrepTile / kPrepThreads;
  __shared__ uint32_t warp_cnt[kSubTiles][kPrepThreads / 32];  // linked anchors per (sub-tile, warp)
  __shared__ uint16_t s_list[kPrepTile];  // the tile's linked anchors (index inside the tile), ascending
  __shared__ uint8_t s_state[kPrepTile];  // 0 final (no predecessor), 0xFF pending, r settled in round r
  if (a.ctr->abort) return;
  const uint32_t n = (uint32_t)a.ctr->n_anchors;  // < 2^30
  const uint32_t tile0 = blockIdx.x * kPrepTile;
  if (tile0 >= n) return;  // the grid is sized for the buffers, not for the count
  const KeyLayout kl = a.kl;
  {
    // all of a thread's key loads first, then the unpacking: five loads in flight instead of one
    // (the wait for a single load before its use was the kernel's largest stall)
    constexpr int kStage = (kPrepHalo + kPrepTile + kPrepThreads - 1) / kPrepThreads;
    uint64_t kreg[kStage];
    unsigned have = 0u;
#pragma unroll
    for (int j = 0; j < kStage; ++j) {
      const int x = threadIdx.x + j * kPrepThreads;
      const long long g = (long long)tile0 - kPrepHalo + x;
      kreg[j] = 0ull;
      if (x < kPrepHalo + kPrepTile && g >= 0 && g < (long long)n) {
        kreg[j] = a.key[g];
        have |= 1u << j;
      }
    }
#pragma unroll
    for (int j = 0; j < kStage; ++j) {
      const int x = threadIdx.x + j * kPrepThreads;
      if (x < kPrepHalo + kPrepTile) {
        const uint64_t k = kreg[j];
        int4 v = make_int4(-1, 0, 0, 0);
        if ((have >> j) & 1u) {
          v.x = (int)(uint32_t)kl.seg(k);
          v.y = (int32_t)kl.target(k);
          v.z = (int32_t)kl.query(k);
        }
        s_a[x] = v;
      }
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned link_mask[kSubTiles];  // my warp's linked lanes, per sub-tile
#pragma unroll
  for (int sub = 0; sub < kSubTiles; ++sub) {
    const int local = sub * kPrepThreads + threadIdx.x;
    const uint32_t i = tile0 + local;
    bool linked = false;
    if (i < n) {
      const int me = kPrepHalo + local;
      const float di = a.dist[i];  // needed after the walk: in flight during it
      const int4 mine = s_a[me];
      const uint32_t sg = (uint32_t)mine.x;
      const int32_t ti = mine.y, qi = mine.z;
      if (sg < a.n_slots) {
        const uint32_t sp = (uint32_t)s_a[me - 1].x;  // 0xFFFFFFFF before the first anchor
        if (i == 0 || sp != sg) {
          a.seg[sg].start = i;
          if (i > 0 && sp < a.n_slots) a.seg[sp].end = i;
        }
        if (i == n - 1) a.seg[sg].end = n;
      }
      // position-only link test over the maximal lookback range, cut where the target gap alone
      // rules every further predecessor out: 3 dt >= 4 (q_i - qmin) >= 4 dq
      const int32_t qlim = sg < a.n_slots ? 4 * (qi - (int32_t)a.seg_qmin[sg]) : 0x7FFFFFFF;
      const int depth = (int)min(i, (uint32_t)kBand);
      const int in_smem = min(depth, me);
      int d = 1;
      bool open = true;  // the range continues past what has been looked at
      for (; d <= in_smem; ++d) {
        const int4 p = s_a[me - d];
        if (p.x != mine.x || p.y + kMaxTargetGap < ti || 3 * (ti - p.y) >= qlim) {
          open = false;
          break;
        }
        if (gap_compatible(ti - p.y, qi - p.z)) {
          linked = true;
          open = false;
          break;
        }
      }
      if (open) {  // rare: deeper than what is staged
        for (; d <= depth; ++d) {
          const uint64_t kj = a.key[i - d];
          const int32_t pt = (int32_t)kl.target(kj);
          if ((uint32_t)kl.seg(kj) != sg || pt + kMaxTargetGap < ti || 3 * (ti - pt) >= qlim) break;
          if (gap_compatible(ti - pt, qi - (int32_t)kl.query(kj))) {
            linked = true;
            break;
          }
        }
      }
      const float ci = distance_coefficient(di, (double)a.radius);
      const float init = __fmul_rn(ci, (float)kDim);
      a.coef[i] = ci;
      a.score[i] = init;
      a.pred[i] = linked ? (i | kPending) : i;
      s_a[me].w = __float_as_int(init);  // phase 1 readers only look at x, y, z
    }
    s_state[local] = linked ? (uint8_t)0xFF : (uint8_t)0;
    link_mask[sub] = __ballot_sync(0xffffffffu, linked);
    if (lane == 0) warp_cnt[sub][wid] = __popc(link_mask[sub]);
  }
  // ordered compaction of the linked anchors: index order is (sub-tile, warp, lane), so one
  // barrier and a walk over the 32 counts place every one of them
  __syncthreads();
  uint32_t at = 0, total = 0;
#pragma unroll
  for (int sub = 0; sub < kSubTiles; ++sub) {
    uint32_t before = 0, sub_total = 0;
#pragma unroll
    for (int w = 0; w < kPrepThreads / 32; ++w) {
      const uint32_t t = warp_cnt[sub][w];
      if (w < wid) before += t;
      sub_total += t;
    }
    const unsigned m = link_mask[sub];
    if (m & (1u << lane)) {
      const uint32_t local = sub * kPrepThreads + threadIdx.x;
      const uint32_t at_list = at + before + __popc(m & ((1u << lane) - 1u));
      a.link_list[(size_t)blockIdx.x * kPrepTile + at_list] = tile0 + local;
      s_list[at_list] = (uint16_t)local;
    }
    at += sub_total;
    total += sub_total;
  }
  if (threadIdx.x == 0) {
    a.link_count[blockIdx.x] = total;
    if (total) atomicAdd(&a.ctr->n_linked, (unsigned long long)total);
  }
  if (total == 0) {
    if (threadIdx.x == 0) a.pend_count[blockIdx.x] = 0;
    return;
  }
  __syncthreads();  // s_list, s_state and the scores are complete

  // ---- phase 2: settle rounds
  for (int round = 1; round <= a.prep_rounds; ++round) {
    for (uint32_t c = threadIdx.x; c < total; c += kPrepThreads) {
      const int local = s_list[c];
      if (s_state[local] != 0xFF) continue;
      const int me = kPrepHalo + local;
      const int4 mine = s_a[me];
      const int32_t ti = mine.y, qi = mine.z;
      const uint32_t i = tile0 + (uint32_t)local;
      const float ci = a.coef[i];
      // no predecessor at or beyond 3 dt >= 4 (q_i - qmin) can be gap-compatible: whatever the
      // reference's loop still does there (count skips, break) leaves score and predecessor as they are
      const int32_t qlim = (uint32_t)mine.x < a.n_slots ? 4 * (qi - (int32_t)a.seg_qmin[mine.x]) : 0x7FFFFFFF;
      float M = __int_as_float(mine.w);  // 6 * coef = chaining_scores[anchor_index]
      uint32_t best = i;
      int S = 0;  // num_skips
      bool defer = false;
      int x = me - 1;
      for (; x >= 0; --x) {
        const int4 p = s_a[x];
        if (p.x != mine.x) break;  // the first anchor of the segment has been passed
        if (3 * (ti - p.y) >= qlim) break;
        if (p.z == qi || p.y == ti) continue;
        if (p.y + kMaxTargetGap < ti) break;
        const int32_t dt = ti - p.y, dq = qi - p.z;
        if (dq < 0) continue;
        float cur = 0.0f;
        if (gap_compatible(dt, dq)) {
          const int pl = x - kPrepHalo;
          if (pl < 0 || s_state[pl] >= (uint32_t)round) {  // halo / pending / being settled right now
            defer = true;
            break;
          }
          cur = __fadd_rn(__int_as_float(p.w), __fmul_rn((float)min(min(dt, dq), kDim), ci));
        }
        if (cur > M) {
          M = cur;
          best = tile0 + (uint32_t)(x - kPrepHalo);
          --S;
        } else if (++S > kMaxSkips) {
          break;
        }
      }
      if (x < 0) defer = true;  // the range goes on before the staged halo
      if (!defer) {
        s_a[me].w = __float_as_int(M);
        s_state[local] = (uint8_t)round;
        a.score[i] = M;
        a.pred[i] = best;  // clears kPending
      }
    }
    __syncthreads();
  }

  // ---- what is still pending, compacted in order, for k_chain_dp / k_dp_pass
  uint32_t pbase = 0;
  for (uint32_t c0 = 0; c0 < total; c0 += kPrepThreads) {
    const uint32_t c = c0 + threadIdx.x;
    const uint32_t local = c < total ? s_list[c] : 0u;
    const bool pend = c < total && s_state[local] == 0xFF;
    const unsigned m = __ballot_sync(0xffffffffu, pend);
    if (lane == 0) warp_cnt[0][wid] = __popc(m);
    __syncthreads();
    uint32_t before = 0, chunk_total = 0;
#pragma unroll
    for (int w = 0; w < kPrepThreads / 32; ++w) {
      const uint32_t t = warp_cnt[0][w];
      if (w < wid) before += t;
      chunk_total += t;
    }
    if (pend) a.pend_list[(size_t)blockIdx.x * kPrepTile + pbase + before + __popc(m & ((1u << lane) - 1u))] = (uint16_t)local;
    pbase += chunk_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    a.pend_count[blockIdx.x] = pbase;
    if (pbase) atomicAdd(&a.ctr->n_pending, (unsigned long long)pbase);
  }
}

constexpr int kDpThreads = 128;
constexpr int kDpFreePasses = 1;  // thread-parallel passes before the in-order cooperative path (measured: 1 < 2 < 4)
constexpr int kDpGroup = 4;       // predecessors fetched together in the thread-parallel lookback

// A warp owns a segment and takes its linked anchors 32 at a time, one per lane.
//  * Thread-parallel passes: every lane runs the reference's lookback for its own anchor.  An
//    anchor's score only depends on the scores of its gap-compatible predecessors; if one of
//    them is still pending (a linked anchor earlier in the same 32) the lane defers, otherwise
//    its result is final.  Background hits form chains of 2-3 anchors, so two passes settle
//    almost everything.
//  * What is still pending after that (true-locus clusters, where every anchor links to the
//    previous one) is settled in order by the whole warp: lanes load 32 consecutive predecessors
//    coalesced, score one each, and the sequential rules (continue/break, running best, +-1 skip
//    counter with its > 25 break) are resolved with a prefix-max scan and ballots.
__device__ __forceinline__ void dp_segment(const ChainArgs &a, const uint32_t slot, const int lane) {
  const unsigned full = 0xffffffffu;
  const unsigned le = (2u << lane) - 1u;  // lanes 0..lane
  SegRec r = a.seg[slot];
  if (r.start == kSegEmpty) return;
  const uint32_t s = r.start, e = r.end;
  const KeyLayout kl = a.kl;
  const uint64_t *key = a.key;
  float *score = a.score;
  uint32_t *pred = a.pred;

  // max over the linked anchors only: the others score <= 6, and every comparison this max
  // feeds has a candidate score >= min_chaining_score = 10 on the other side (:545-567)
  float runmax = 0.0f;
  float ts0 = 0.f, ts1 = 0.f, ts2 = 0.f;  // best three local end candidates
  uint32_t ti0 = 0, ti1 = 0, ti2 = 0;
  int ntop = 0;

  for (uint32_t tile = s / kPrepTile; tile * kPrepTile < e; ++tile) {
    // ---- phase A: the lookback for the anchors k_chain_prep (and k_dp_pass) left pending
    const uint32_t pcnt = a.pend_count[tile];
    const uint16_t *plist = a.pend_list + (size_t)tile * kPrepTile;
    for (uint32_t c0 = 0; c0 < pcnt; c0 += 32) {
      const uint32_t c = c0 + lane;
      uint32_t i = c < pcnt ? tile * kPrepTile + (uint32_t)plist[c] : 0xFFFFFFFFu;
      const bool valid = c < pcnt && i >= s && i < e && (pred[i] & kPending);
      if (!__ballot_sync(full, valid)) continue;
      int32_t ti = 0, qi = 0;
      float ci = 0.0f, init = 0.0f, M = 0.0f;
      uint32_t lo = 0;
      if (valid) {
        const uint64_t k = key[i];
        ti = (int32_t)kl.target(k);
        qi = (int32_t)kl.query(k);
        ci = a.coef[i];
        init = score[i];  // still 6 * coef from k_chain_prep = chaining_scores[anchor_index]
        lo = (i - s > (uint32_t)kBand) ? i - kBand : s;
      }
      bool todo = valid;
      // ---- thread-parallel passes
      for (int pass = 0; pass < a.dp_passes; ++pass) {
        if (todo) {
          M = init;
          uint32_t best = i;
          int S = 0;  // num_skips
          bool defer = false;
          // predecessors four at a time: the key loads of a group are independent, so the walk
          // pays one memory round trip per group instead of one per predecessor
          bool done = false;
          for (uint32_t jb = i; jb > lo && !done;) {
            const uint32_t m = min(jb - lo, (uint32_t)kDpGroup);
            uint64_t kk[kDpGroup];
#pragma unroll
            for (int u = 0; u < kDpGroup; ++u) kk[u] = (uint32_t)u < m ? key[jb - 1u - (uint32_t)u] : 0ull;
#pragma unroll
            for (int u = 0; u < kDpGroup; ++u) {
              if (done || (uint32_t)u >= m) break;
              const uint32_t j = jb - 1u - (uint32_t)u;
              const uint64_t kj = kk[u];
              const int32_t pt = (int32_t)kl.target(kj), pq = (int32_t)kl.query(kj);
              if (pq == qi || pt == ti) continue;
              if (pt + kMaxTargetGap < ti) {
                done = true;
                break;
              }
              const int32_t dt = ti - pt, dq = qi - pq;
              if (dq < 0) continue;
              float cur = 0.0f;
              if (gap_compatible(dt, dq)) {
                if (pred[j] & kPending) {
                  defer = true;
                  done = true;
                  break;
                }
                cur = __fadd_rn(score[j], __fmul_rn((float)min(min(dt, dq), kDim), ci));
              }
              if (cur > M) {
                M = cur;
                best = j;
                --S;
              } else if (++S > kMaxSkips) {
                done = true;
                break;
              }
            }
            jb -= m;
          }
          if (!defer) {
            score[i] = M;
            pred[i] = best;  // clears kPending
            todo = false;
          }
        }
        __syncwarp(full);  // settled scores are visible to the lanes that deferred
        if (!__ballot_sync(full, todo)) break;
      }
      // ---- what is left, in order, by the whole warp
      unsigned left = __ballot_sync(full, todo);
      while (left) {
        const int src = __ffs(left) - 1;
        left &= left - 1;
        const uint32_t ii = __shfl_sync(full, i, src);
        const int32_t tii = __shfl_sync(full, ti, src), qii = __shfl_sync(full, qi, src);
        const float cii = __shfl_sync(full, ci, src);
        const uint32_t loi = __shfl_sync(full, lo, src);
        float Mi = __shfl_sync(full, init, src);
        uint32_t best = ii;
        int S = 0;
        for (uint32_t jb = ii;; jb -= 32) {  // block of predecessors jb-1 .. jb-32
          // ---- my predecessor: >= 0 candidate score (counted), -1 continue, -2 lookback ends
          float cd = -2.0f;
          if (jb >= loi + 1u + (uint32_t)lane) {
            const uint32_t j = jb - 1u - (uint32_t)lane;
            const uint64_t kj = key[j];
            const int32_t pt = (int32_t)kl.target(kj), pq = (int32_t)kl.query(kj);
            const int32_t dt = tii - pt, dq = qii - pq;
            if (pq == qii || pt == tii) cd = -1.0f;
            else if (pt + kMaxTargetGap < tii) cd = -2.0f;
            else if (dq < 0) cd = -1.0f;
            else if (gap_compatible(dt, dq)) cd = __fadd_rn(score[j], __fmul_rn((float)min(min(dt, dq), kDim), cii));
            else cd = 0.0f;
          }
          // ---- resolve the 32 predecessors in order (lane 0 = most recent)
          const bool counted = cd >= 0.0f;
          const unsigned cntm = __ballot_sync(full, counted);
          unsigned impm = 0u;
          if (__ballot_sync(full, cd > Mi)) {
            float pm = counted ? cd : 0.0f;  // inclusive prefix max of the candidate scores
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
              const float t = __shfl_up_sync(full, pm, d);
              if (lane >= d) pm = fmaxf(pm, t);
            }
            float ex = __shfl_up_sync(full, pm, 1);
            ex = fmaxf(lane == 0 ? 0.0f : ex, Mi);
            impm = __ballot_sync(full, counted && cd > ex);
          }
          const int Sl = S + __popc(cntm & ~impm & le) - __popc(impm & le);
          const bool stop_here = (counted && !((impm >> lane) & 1u) && Sl > kMaxSkips) || cd == -2.0f;
          const unsigned stopm = __ballot_sync(full, stop_here);
          const unsigned below = stopm ? ((stopm & (0u - stopm)) - 1u) : full;
          const unsigned imp_b = impm & below;
          if (imp_b) {
            const int L = 31 - __clz(imp_b);
            Mi = __shfl_sync(full, cd, L);
            best = jb - 1u - (uint32_t)L;
          }
          if (stopm) break;
          S += __popc(cntm & ~impm) - __popc(impm);
        }
        if (lane == src) {
          M = Mi;
          score[ii] = Mi;
          pred[ii] = best;
        }
        __syncwarp(full);  // visible to the later anchors of this batch
      }
    }
    // ---- phase B: running max and local end candidates (spatial_index.cc:542-549) over ALL linked
    // anchors of the tile, lanes in order; the caller applies the max of the earlier buckets, which
    // only shortens this list.  Order: score desc, index desc (compare(), :11-20); a tie puts the
    // later anchor first.
    __syncwarp(full);
    const uint32_t cnt = a.link_count[tile];
    const uint32_t *list = a.link_list + (size_t)tile * kPrepTile;
    // four batches of 32 per round trip: the list entries, then their scores, are loaded together
    for (uint32_t c0 = 0; c0 < cnt; c0 += 128) {
      uint32_t iv[4];
      float Mv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t c = c0 + 32u * (uint32_t)u + lane;
        iv[u] = c < cnt ? list[c] : 0xFFFFFFFFu;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (iv[u] < s || iv[u] >= e) iv[u] = 0xFFFFFFFFu;  // another segment's anchor
        Mv[u] = iv[u] != 0xFFFFFFFFu ? score[iv[u]] : 0.0f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const bool valid = iv[u] != 0xFFFFFFFFu;
        if (!__ballot_sync(full, valid)) continue;
        const uint32_t i = iv[u];
        const float M = Mv[u];
        float pm = M;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const float t = __shfl_up_sync(full, pm, d);
          if (lane >= d) pm = fmaxf(pm, t);
        }
        pm = fmaxf(pm, runmax);
        unsigned candm = __ballot_sync(full, valid && M >= 10.0f && M > __fdiv_rn(pm, 2.0f));
        runmax = __shfl_sync(full, pm, 31);
        while (candm) {
          const int l = __ffs(candm) - 1;
          candm &= candm - 1;
          const float Ml = __shfl_sync(full, M, l);
          const uint32_t il = __shfl_sync(full, i, l);
          if (ntop < 1 || Ml >= ts0) {
            ts2 = ts1; ti2 = ti1; ts1 = ts0; ti1 = ti0; ts0 = Ml; ti0 = il;
            if (ntop < 3) ++ntop;
          } else if (ntop < 2 || Ml >= ts1) {
            ts2 = ts1; ti2 = ti1; ts1 = Ml; ti1 = il;
            if (ntop < 3) ++ntop;
          } else if (ntop < 3 || Ml >= ts2) {
            ts2 = Ml; ti2 = il;
            if (ntop < 3) ++ntop;
          }
        }
      }
    }
  }
  if (lane == 0) {
    r.ntop = (uint32_t)ntop;
    r.max = runmax;
    r.top_s[0] = ts0; r.top_s[1] = ts1; r.top_s[2] = ts2;
    r.top_i[0] = ti0; r.top_i[1] = ti1; r.top_i[2] = ti2;
    a.seg[slot] = r;
    a.seg_max[slot] = runmax;
  }
}

// ---- small batches (read-until rounds): the same lookback for every linked anchor of the step at
// once.  With a few hundred chunks there are only a few hundred segments, and a warp walking a
// segment's ~1 500 linked anchors 32 at a time is a 50-step serial chain: the round's latency.
// Here persistent warps take k_chain_prep TILES instead, so the anchors of one segment are walked
// by many warps at once.  An anchor's score only depends on the scores of its gap-compatible
// predecessors; if the lookback meets one that is still pending the lane defers (<= 3 tries, then
// it is left to the in-order kernel), otherwise its result is final whatever other warps are doing,
// so results do not depend on timing.  Scores of other warps' anchors are read past L1 (ld.cg)
// after their pending bit was seen cleared; the writer orders score before bit with a fence.  On
// large batches this loses to the in-segment pass (every cross-warp score is an L2 round trip in
// the middle of a walk; measured 7 ms against 5.5 ms on 360 M anchors), so the host only launches
// it up to kDpPassMaxEntries chunks per step (the segments of one chunk are what a warp of the
// in-segment kernel would walk alone, however many buckets the reference has).
constexpr int kDpPassThreads = 256;
constexpr uint32_t kDpPassMaxEntries = 4096;
constexpr int kDpIters = 3;      // tries per anchor inside its warp before it is left to the in-order kernel

__global__ void __launch_bounds__(kDpPassThreads, 6) k_dp_pass(ChainArgs a) {
  if (a.ctr->abort) return;
  const uint32_t n = (uint32_t)a.ctr->n_anchors;
  const uint32_t n_tiles = (n + kPrepTile - 1) / kPrepTile;
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * kDpPassThreads + threadIdx.x) >> 5;
  const uint32_t n_warps = (gridDim.x * kDpPassThreads) >> 5;
  const unsigned full = 0xffffffffu;
  const KeyLayout kl = a.kl;
  const uint64_t *__restrict__ key = a.key;
  float *score = a.score;
  uint32_t *pred = a.pred;
  for (uint32_t tile = warp; tile < n_tiles; tile += n_warps) {
    const uint32_t cnt = a.pend_count[tile];
    const uint16_t *list = a.pend_list + (size_t)tile * kPrepTile;
    for (uint32_t c0 = 0; c0 < cnt; c0 += 32) {
      const uint32_t c = c0 + lane;
      const bool have = c < cnt;
      const uint32_t i = have ? tile * kPrepTile + (uint32_t)list[c] : 0u;
      bool todo = have && (__ldcg(pred + i) & kPending);
      uint64_t sg = 0;
      int32_t ti = 0, qi = 0;
      float ci = 0.0f, init = 0.0f;
      if (todo) {
        const uint64_t k = key[i];
        sg = kl.seg(k);
        ti = (int32_t)kl.target(k);
        qi = (int32_t)kl.query(k);
        ci = a.coef[i];
        init = __ldcg(score + i);  // 6 * coef from k_chain_prep = chaining_scores[anchor_index]
      }
      for (int iter = 0; iter < kDpIters && __any_sync(full, todo); ++iter) {
        if (todo) {
          float M = init;
          uint32_t best = i;
          int S = 0;  // num_skips
          bool defer = false, done = false;
          const uint32_t lo = i > (uint32_t)kBand ? i - kBand : 0u;  // the segment start ends the walk earlier
          // predecessors four at a time: the key loads of a group are independent, so the walk
          // pays one memory round trip per group instead of one per predecessor
          for (uint32_t jb = i; jb > lo && !done;) {
            const uint32_t m = min(jb - lo, (uint32_t)kDpGroup);
            uint64_t kk[kDpGroup];
#pragma unroll
            for (int u = 0; u < kDpGroup; ++u) kk[u] = (uint32_t)u < m ? key[jb - 1u - (uint32_t)u] : 0ull;
#pragma unroll
            for (int u = 0; u < kDpGroup; ++u) {
              if (done || (uint32_t)u >= m) break;
              const uint32_t j = jb - 1u - (uint32_t)u;
              const uint64_t kj = kk[u];
              if (kl.seg(kj) != sg) {  // first anchor of the segment passed
                done = true;
                break;
              }
              const int32_t pt = (int32_t)kl.target(kj), pq = (int32_t)kl.query(kj);
              if (pq == qi || pt == ti) continue;
              if (pt + kMaxTargetGap < ti) {
                done = true;
                break;
              }
              const int32_t dt = ti - pt, dq = qi - pq;
              if (dq < 0) continue;
              float cur = 0.0f;
              if (gap_compatible(dt, dq)) {
                if (__ldcg(pred + j) & kPending) {
                  defer = true;
                  done = true;
                  break;
                }
                cur = __fadd_rn(__ldcg(score + j), __fmul_rn((float)min(min(dt, dq), kDim), ci));
              }
              if (cur > M) {
                M = cur;
                best = j;
                --S;
              } else if (++S > kMaxSkips) {
                done = true;
                break;
              }
            }
            jb -= m;
          }
          if (!defer) {
            score[i] = M;
            __threadfence();
            pred[i] = best;  // clears kPending
            todo = false;
          }
        }
        __syncwarp(full);
      }
    }
  }
}


// Segments differ a lot in how many linked anchors they hold, so a fixed warp <-> segment
// assignment leaves most warps of a block idle behind its slowest one: persistent warps take
// segments from a work cursor instead.
__global__ void __launch_bounds__(kDpThreads) k_chain_dp(ChainArgs a) {
  const int lane = threadIdx.x & 31;
  if (a.ctr->abort) return;
  for (;;) {
    uint32_t slot = 0;
    if (lane == 0) slot = atomicAdd(&a.ctr->dp_cursor, 1u);
    slot = __shfl_sync(0xffffffffu, slot, 0);
    if (slot >= a.n_slots) break;
    dp_segment(a, slot, lane);
  }
}

// ---------------------------------------------------------------------------------------
// K7: chains and the per-read decision, in two kernels with an optional exchange in between
// (contig-sharded index, SURVEY.md 8e mode 2: the buckets of one read live on several GPUs).
//
//   k_sel_trace   warp per (entry, bucket) segment: the running max of the EARLIER buckets
//                 (spatial_index.cc:419, a prefix max over seg_max[], which a sharded run
//                 all-reduces first), then TracebackChains (spatial_index.cc:165-220) for the
//                 segment's <= 3 end candidates.  The walk keeps a 32-anchor window of pred[]
//                 in registers (one lane each) and follows the chain with shuffles: chain
//                 members are near neighbours in the sorted order, so a window serves 20-30
//                 steps and the walk issues ~25x fewer dependent global loads than a
//                 thread-per-read pointer chase.  Visited anchors are written, end -> start,
//                 to path[], so later copies are parallel gathers.
//   k_sel_scatter (sharded only) candidates gathered from the other ranks join the per-entry
//                 lists.
//   k_sel_pick    warp per entry: GeneratePrimaryChains (spatial_index.cc:222-253) on lane 0 and
//                 the carry-pool space the survivors need (nothing committed yet)
//   k_sel_commit  warp per entry: ComputeMAPQ (:255-274), all lanes copy the surviving chains'
//                 anchors to the carry pool (only chains whose bucket this rank owns), the
//                 StreamingMap stop / output decision and the tag sums (sigmap.cc:667-745).
struct CandRec {  // an end candidate whose traceback produced a chain of >= 2 anchors
  float score;
  uint32_t entry, bucket, start, end, n;
  uint32_t end_idx;   // anchor index of the chain end (owner rank's arrays)
  uint32_t path_off;  // first of n path[] entries (owner rank's arrays)
  uint32_t owner;     // rank whose index shard holds the bucket
};

struct ChainTmp {
  CandRec c;
  uint32_t state;  // 0 candidate, 1 primary (order in `rank`), 2 rejected
  uint32_t rank;
  uint32_t order;  // record r: index of the primary chain of rank r (k_sel_pick -> k_sel_commit)
};

struct SelectArgs {
  ChainArgs c;
  const uint32_t *entry_slot;
  const uint32_t *n_queries;   // 0 => GenerateChains not called (copy state forward)
  const uint32_t *n_features;
  SlotState *slots;
  uint32_t B;
  ChainTmp *scratch;           // [B][max_chains]
  uint32_t *n_scratch;         // [B] candidates per entry (zeroed before k_sel_trace)
  uint32_t max_chains;
  uint32_t *path;              // [n] traceback paths, a segment's chains packed from seg.start
  CandRec *cand_list;          // sharded: compact list of this rank's candidates (else nullptr)
  uint32_t cand_cap;
  uint32_t rank;               // this rank (0 when not sharded)
  uint32_t out_pool;
  ChainRec *pool_chain[2];
  CarryAnchor *pool_anchor[2];
  unsigned long long pool_chain_cap, pool_anchor_cap;
  smb_params prm;
};

constexpr int kTraceThreads = 128;
constexpr uint32_t kUsed = 0x80000000u;  // pred[] bit: anchor_is_used (spatial_index.cc:170)

__device__ __forceinline__ void add_candidate(const SelectArgs &a, const CandRec &c) {
  const uint32_t at = atomicAdd(&a.n_scratch[c.entry], 1u);
  if (at < a.max_chains) {
    ChainTmp t;
    t.c = c;
    t.state = 0;
    t.rank = 0;
    t.order = 0;
    a.scratch[(size_t)c.entry * a.max_chains + at] = t;
  } else {
    atomicOr(&a.c.ctr->error, 4u);
  }
}

__global__ void __launch_bounds__(kTraceThreads) k_sel_trace(SelectArgs a) {
  const int lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  const uint32_t slot = (blockIdx.x * kTraceThreads + threadIdx.x) / 32;
  if (slot >= a.c.n_slots || a.c.ctr->abort) return;
  const SegRec rec = a.c.seg[slot];
  if (rec.start == kSegEmpty || rec.ntop == 0u || rec.ntop > 3u) return;
  const KeyLayout kl = a.c.kl;
  const uint32_t bucket = slot & ((1u << kl.bbits) - 1u), entry = slot >> kl.bbits;
  const uint32_t n = (uint32_t)a.c.ctr->n_anchors;
  uint32_t *pred = a.c.pred;
  const float *score = a.c.score;

  // max_chaining_score before this bucket (buckets in the reference's order, :420-422)
  float gprev = 0.0f;
  for (uint32_t k = lane; k < bucket; k += 32) gprev = fmaxf(gprev, a.c.seg_max[slot - bucket + k]);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) gprev = fmaxf(gprev, __shfl_xor_sync(full, gprev, d));
  // The DP kept the segment's best three end candidates under its own running max; the
  // reference's test also includes the earlier buckets' max, which removes exactly the
  // candidates with score <= gprev/2 -- a suffix of the list (:545-549).
  const float half_prev = __fdiv_rn(gprev, 2.0f);
  const float half = __fdiv_rn(fmaxf(gprev, rec.max), 2.0f);

  uint32_t path_at = rec.start;
  for (uint32_t r = 0; r < rec.ntop; ++r) {
    if (!(rec.top_s[r] > half_prev)) break;
    const uint32_t e = rec.top_i[r];
    // ---- TracebackChains (spatial_index.cc:165-220) over a register window of pred[]
    uint32_t wlo = e >= 31u ? e - 31u : 0u;
    uint32_t v = (wlo + lane < n) ? pred[wlo + lane] : 0u;
    bool dirty = false;
    if (!(__shfl_sync(full, v, (int)(e - wlo)) & kUsed)) {
      uint32_t s = e, cnt = 0, stop_pred = e;
      bool hit_used = false;
      for (;;) {
        const uint32_t p = __shfl_sync(full, v, (int)(s - wlo)) & 0x3FFFFFFFu;
        if ((uint32_t)lane == s - wlo) {
          v |= kUsed;
          dirty = true;
        }
        if (lane == 0) a.path[path_at + cnt] = s;
        ++cnt;
        if (p == s) break;  // chain start: its own predecessor
        if (p < wlo) {      // slide the window so that p is its last element
          if (dirty) pred[wlo + lane] = v;
          dirty = false;
          __syncwarp(full);
          wlo = p >= 31u ? p - 31u : 0u;
          v = (wlo + lane < n) ? pred[wlo + lane] : 0u;
        }
        if (__shfl_sync(full, v, (int)(p - wlo)) & kUsed) {
          hit_used = true;
          stop_pred = p;
          break;
        }
        s = p;
      }
      if (dirty) pred[wlo + lane] = v;
      __syncwarp(full);
      if (cnt >= 2u && lane == 0) {
        CandRec c;
        c.score = score[e];
        if (hit_used) c.score = __fsub_rn(c.score, score[stop_pred]);
        c.entry = entry;
        c.bucket = bucket;
        c.start = kl.target(a.c.key[s]);
        c.end = kl.target(a.c.key[e]);
        c.n = cnt;
        c.end_idx = e;
        c.path_off = path_at;
        c.owner = a.rank;
        add_candidate(a, c);
        if (a.cand_list) {
          const unsigned long long at = atomicAdd(&a.c.ctr->n_cand, 1ull);
          if (at < a.cand_cap) a.cand_list[at] = c;
          else atomicOr(&a.c.ctr->error, 32u);
        }
      }
      if (cnt >= 2u) path_at += cnt;
    }
    if (score[e] < half) break;  // :564-567
  }
}

// sharded: candidates of the other ranks (gathered lists, `per_rank` records each) join the
// per-entry scratch lists; the order inside a list is irrelevant (the selection below is a
// total order on (score, n, dir, contig, start, end)).
__global__ void k_sel_scatter(SelectArgs a, const CandRec *__restrict__ all, const unsigned long long *__restrict__ counts,
                              uint32_t world, uint32_t per_rank) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t r = i / per_rank, k = i % per_rank;
  if (r >= world || r == a.rank || k >= counts[r] || a.c.ctr->abort) return;
  add_candidate(a, all[(size_t)r * per_rank + k]);
}

// spatial_index.h:38-44 operator> on (score, n, dir, contig, start, end)
__device__ __forceinline__ bool chain_greater(const CandRec &x, const CandRec &y) {
  if (x.score != y.score) return x.score > y.score;
  if (x.n != y.n) return x.n > y.n;
  const uint32_t xd = (x.bucket & 1u) ^ 1u, yd = (y.bucket & 1u) ^ 1u;  // strand bit 0 = Positive (enum 1)
  if (xd != yd) return xd > yd;
  if ((x.bucket >> 1) != (y.bucket >> 1)) return (x.bucket >> 1) > (y.bucket >> 1);
  if (x.start != y.start) return x.start > y.start;
  return x.end > y.end;
}

constexpr int kFinalThreads = 128;

// what k_sel_pick decided for one entry
struct PickRec {
  uint32_t n_prim, prim_first, prim_second, total_anchors;
};

// warp per entry: GeneratePrimaryChains (spatial_index.cc:222-253) on the entry's candidate list,
// and the carry-pool space the survivors will need.  Nothing is committed here: the pools are
// checked against the step's total need (k_pool_check) before k_sel_commit writes anything, so a
// step whose survivors do not fit can be redone with larger pools.
__global__ void __launch_bounds__(kFinalThreads) k_sel_pick(SelectArgs a, PickRec *__restrict__ pick) {
  const int lane = threadIdx.x & 31;
  const uint32_t b = (blockIdx.x * kFinalThreads + threadIdx.x) / 32;
  if (b >= a.B || a.c.ctr->abort) return;
  Counters *ctr = a.c.ctr;
  if (a.n_queries[b] == 0) {  // chains unchanged: they move to the pool that survives the round
    if (lane == 0) {
      const SlotState &st = a.slots[a.entry_slot[b]];
      if (st.n_chains > 0) {
        atomicAdd(&ctr->need_chain, (unsigned long long)st.n_chains);
        atomicAdd(&ctr->need_anchor, (unsigned long long)st.carry_n);
      }
    }
    return;
  }
  // The reference sorts the candidates in descending order and walks them (:222-253); here the
  // maximum is extracted again and again by the whole warp: every lane scans its share of the
  // candidates, a shuffle tournament under the reference's order (ties: the lower index, which is
  // what a sequential first-maximum scan keeps) picks the next one, and the overlap test against the
  // primaries found so far is shared the same way.  A weak first chain lets every candidate through
  // the score test, so one lane alone paid candidates^2 dependent loads (1.4 ms of a read-until round
  // on a 32-bucket reference).
  const unsigned full = 0xffffffffu;
  ChainTmp *ch = a.scratch + (size_t)b * a.max_chains;
  const uint32_t nch = min(a.n_scratch[b], a.max_chains);
  uint32_t n_prim = 0, prim_first = 0, prim_second = 0, total_anchors = 0;
  float last_primary_score = 0.0f;
  for (;;) {
    int best = -1;
    CandRec bc{};
    for (uint32_t c = lane; c < nch; c += 32) {
      if (ch[c].state != 0) continue;
      const CandRec cc = ch[c].c;
      if (best < 0 || chain_greater(cc, bc)) {
        best = (int)c;
        bc = cc;
      }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      CandRec oc = bc;
      const int ob = __shfl_xor_sync(full, best, d);
      oc.score = __shfl_xor_sync(full, bc.score, d);
      oc.n = __shfl_xor_sync(full, bc.n, d);
      oc.bucket = __shfl_xor_sync(full, bc.bucket, d);
      oc.start = __shfl_xor_sync(full, bc.start, d);
      oc.end = __shfl_xor_sync(full, bc.end, d);
      if (ob >= 0 && (best < 0 || chain_greater(oc, bc) || (!chain_greater(bc, oc) && ob < best))) {
        best = ob;
        bc.score = oc.score;
        bc.n = oc.n;
        bc.bucket = oc.bucket;
        bc.start = oc.start;
        bc.end = oc.end;
      }
    }
    if (best < 0) break;
    const CandRec cb = ch[best].c;  // the same record on every lane
    if (n_prim > 0 && cb.score < __fdiv_rn(last_primary_score, 3.0f)) break;
    bool clash = false;
    for (uint32_t c = lane; c < nch; c += 32) {
      if (ch[c].state != 1 || (ch[c].c.bucket >> 1) != (cb.bucket >> 1)) continue;
      const uint32_t mx = max(cb.start, ch[c].c.start), mn = min(cb.end, ch[c].c.end);
      if (!(mx > mn)) clash = true;
    }
    const bool ok = !__any_sync(full, clash);
    if (lane == 0) {
      if (ok) {
        ch[best].state = 1;
        ch[best].rank = n_prim;
        ch[n_prim].order = (uint32_t)best;
      } else {
        ch[best].state = 2;
      }
    }
    if (ok) {
      if (n_prim == 0) prim_first = (uint32_t)best;
      if (n_prim == 1) prim_second = (uint32_t)best;
      last_primary_score = cb.score;
      if (cb.owner == a.rank) total_anchors += cb.n;
      ++n_prim;
    }
    __syncwarp(full);  // the new state is visible to every lane's next scan
  }
  if (lane == 0) {
    pick[b] = PickRec{n_prim, prim_first, prim_second, total_anchors};
    if (n_prim) {
      atomicAdd(&ctr->need_chain, (unsigned long long)n_prim);
      atomicAdd(&ctr->need_anchor, (unsigned long long)total_anchors);
    }
  }
}

__global__ void k_pool_check(Counters *ctr, uint32_t op, unsigned long long cap_chain, unsigned long long cap_anchor) {
  if (ctr->carry_chain_used[op] + ctr->need_chain > cap_chain || ctr->carry_anchor_used[op] + ctr->need_anchor > cap_anchor)
    ctr->abort |= kAbortPool;
}

// warp per entry: the survivors' records and anchors go to the carry pool, ComputeMAPQ
// (spatial_index.cc:255-274), then StreamingMap's stop / output decision and the tag sums
// (sigmap.cc:667-745) into the read slot.
__global__ void __launch_bounds__(kFinalThreads) k_sel_commit(SelectArgs a, const PickRec *__restrict__ pick) {
  const int lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  const uint32_t b = (blockIdx.x * kFinalThreads + threadIdx.x) / 32;
  if (b >= a.B || a.c.ctr->abort) return;
  const uint32_t slot = a.entry_slot[b];
  SlotState st = a.slots[slot];
  const uint32_t op = a.out_pool;
  Counters *ctr = a.c.ctr;

  if (a.n_queries[b] == 0) {
    // chains unchanged (chunk skipped: <= 50 features, or no chunk this round); move the
    // slot's records to the pool that survives the next round
    if (st.n_chains > 0) {
      unsigned long long co = 0, ao = 0;
      if (lane == 0) {
        co = atomicAdd(&ctr->carry_chain_used[op], (unsigned long long)st.n_chains);
        ao = atomicAdd(&ctr->carry_anchor_used[op], (unsigned long long)st.carry_n);
      }
      co = __shfl_sync(full, co, 0);
      ao = __shfl_sync(full, ao, 0);
      const ChainRec *sc = a.pool_chain[st.pool] + st.chain_off;
      const CarryAnchor *sa = a.pool_anchor[st.pool] + st.carry_off;
      for (uint32_t i = lane; i < st.n_chains; i += 32) a.pool_chain[op][co + i] = sc[i];
      for (uint32_t i = lane; i < st.carry_n; i += 32) a.pool_anchor[op][ao + i] = sa[i];
      st.chain_off = co;
      st.carry_off = ao;
    }
    st.pool = op;
    st.stop = 0;
    if (lane == 0) a.slots[slot] = st;
    return;
  }

  const KeyLayout kl = a.c.kl;
  ChainTmp *ch = a.scratch + (size_t)b * a.max_chains;
  if (a.n_scratch[b] > a.max_chains) st.flags |= 2u;
  const PickRec pk = pick[b];
  const uint32_t n_prim = pk.n_prim, prim_first = pk.prim_first, prim_second = pk.prim_second;
  const uint32_t total_anchors = pk.total_anchors;

  // ---- survivors to the carry pool, primary order, anchors end -> start
  unsigned long long co = 0, ao = 0;
  if (n_prim > 0) {
    if (lane == 0) {
      co = atomicAdd(&ctr->carry_chain_used[op], (unsigned long long)n_prim);
      ao = atomicAdd(&ctr->carry_anchor_used[op], (unsigned long long)total_anchors);
    }
    co = __shfl_sync(full, co, 0);
    ao = __shfl_sync(full, ao, 0);
  }
  float mean = 0.0f;
  uint32_t mapq0 = 0;
  if (n_prim == 1) {
    mapq0 = 60;  // spatial_index.cc:255-258
  } else if (n_prim >= 2) {
    const float ratio = __fdiv_rn(ch[prim_second].c.score, ch[prim_first].c.score);
    int mq = (int)__fmul_rn(40.0f, __fsub_rn(1.0f, ratio));
    mq = mq > 60 ? 60 : (mq < 0 ? 0 : mq);
    mapq0 = (uint32_t)(uint8_t)mq;
  }
  if (n_prim > 0) {
    uint32_t aoff = 0;
    for (uint32_t r = 0; r < n_prim; ++r) {  // ranks are 0..n_prim-1; emit in rank order
      const uint32_t c = ch[r].order;
      const CandRec cc = ch[c].c;
      mean = __fadd_rn(mean, cc.score);
      const bool owned = cc.owner == a.rank;
      if (lane == 0) {
        ChainRec rec;
        rec.score = cc.score;
        rec.contig = cc.bucket >> 1;
        rec.start = cc.start;
        rec.end = cc.end;
        rec.n_anchors = cc.n;
        rec.mapq = r == 0 ? mapq0 : 0;
        rec.dir = (cc.bucket & 1u) ^ 1u;
        rec.anchor_off = owned ? aoff : 0xFFFFFFFFu;
        a.pool_chain[op][co + r] = rec;
      }
      if (owned) {
        CarryAnchor *dst = a.pool_anchor[op] + ao + aoff;
        for (uint32_t k = lane; k < cc.n; k += 32) {
          const uint32_t idx = a.path[cc.path_off + k];
          const uint64_t kk = a.c.key[idx];
          CarryAnchor ca;
          ca.target = kl.target(kk);
          ca.query = kl.query(kk);
          ca.dist = a.c.dist[idx];
          ca.bucket = cc.bucket;
          dst[k] = ca;
        }
        aoff += cc.n;
      }
    }
    mean = __fdiv_rn(mean, (float)n_prim);
  }
  __syncwarp(full);

  // ---- StreamingMap decision + tag sums on chains[0] (sigmap.cc:667-687, :701-745)
  st.n_chains = n_prim;
  st.chain_off = co;
  st.carry_off = ao;
  st.carry_n = total_anchors;
  st.pool = op;
  st.num_events += a.n_features[b];  // sigmap.cc:666
  st.stop = 0;
  st.mapped = 0;
  st.cm = 0;
  st.owned0 = 0;
  st.s1 = st.s2 = st.sm = st.ad = st.at = st.aq = 0.0f;
  st.q_first = st.q_last = 0;
  if (n_prim > 0) {
    const CandRec c0 = ch[prim_first].c;
    const float s0 = c0.score;
    const float s1 = n_prim > 1 ? ch[prim_second].c.score : 0.0f;
    if (c0.owner == a.rank) {
      // sequential fp32 sums in anchor order (sigmap.cc:735-743), values fetched 32 at a time
      const CarryAnchor *an = a.pool_anchor[op] + ao;  // chain 0 is first
      float ad = 0.0f, at = 0.0f, aq = 0.0f;
      for (uint32_t k0 = 0; k0 < c0.n; k0 += 32) {
        const uint32_t k = k0 + lane;
        float d = 0.0f, dt = 0.0f, dq = 0.0f;
        if (k < c0.n) {
          const CarryAnchor x = an[k];
          d = x.dist;
          if (k + 1 < c0.n) {
            const CarryAnchor y = an[k + 1];
            dt = (float)(uint32_t)(x.target - y.target);
            dq = (float)(uint32_t)(x.query - y.query);
          }
        }
        const int m = (int)min(32u, c0.n - k0);
        for (int j = 0; j < m; ++j) {
          ad = __fadd_rn(ad, __shfl_sync(full, d, j));
          if (k0 + j + 1 < c0.n) {
            at = __fadd_rn(at, __shfl_sync(full, dt, j));
            aq = __fadd_rn(aq, __shfl_sync(full, dq, j));
          }
        }
      }
      st.ad = __fdiv_rn(ad, (float)c0.n);
      st.at = __fdiv_rn(at, (float)c0.n);
      st.aq = __fdiv_rn(aq, (float)c0.n);
      st.q_first = an[0].query;
      st.q_last = an[c0.n - 1].query;
      st.owned0 = 1;
    }
    st.s1 = s0;
    st.s2 = s1;
    st.sm = mean;
    st.cm = c0.n;
    st.c0_contig = c0.bucket >> 1;
    st.c0_start = c0.start;
    st.c0_end = c0.end;
    st.c0_dir = (c0.bucket & 1u) ^ 1u;
    st.c0_mapq = mapq0;
    if (n_prim >= 2) {
      const float ratio = __fdiv_rn(s0, s1);
      if (ratio >= a.prm.stop_mapping || s0 >= __fmul_rn(a.prm.stop_mapping_mean, mean)) st.stop = 1;
      if (ratio >= a.prm.stop_mapping_output || s0 >= __fmul_rn(a.prm.stop_mapping_mean_output, mean))
        st.mapped = 1;
    } else {
      if (c0.n >= (uint32_t)a.prm.min_num_anchors) st.stop = 1;
      if (c0.n >= (uint32_t)a.prm.min_num_anchors_output) st.mapped = 1;
    }
  }
  if (lane == 0) a.slots[slot] = st;
}

}  // namespace sb
#endif
