// sb_engine.cu -- the context, the batched pipeline step, the read scheduler, streaming, the
// stage hooks and the rest of the C ABI of include/sigmap_b200.h.  Index construction (every
// smb_index_* and smb_point_cloud_* entry point) is in sb_index.cu; the context is in sb_ctx.cuh.
//
// Execution model (replaces the OpenMP taskloop of sigmap.cc:618-632): instead of one host
// thread walking one read chunk by chunk, all still-active reads advance together in ROUNDS;
// round k maps chunk k of every active read as one batch (split into steps that fit the
// anchor buffers):
//   events (lookahead blocks on their own stream) -> query table -> carry re-injection +
//   radius search -> per-entry shared-memory sort by (bucket, target, query) -> chain prep ->
//   chaining DP -> traceback -> per-read selection/decision.
// The only host<->device traffic per step is a counter readback (anchor count) and, per
// round, 12 bytes per active read (stop flag, kept events, chain count).
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <optional>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <string>
#include <vector>

#include "k_chain.cuh"
#include "k_sort.cuh"
#include "k_events.cuh"
#include "k_index.cuh"
#include "sb_ctx.cuh"

static_assert(kCarryMaxParts == kMaxParts, "one part limit for every run producer");

namespace {
thread_local std::string g_create_error;

inline int bits_for(uint64_t max_value) {  // bits needed to represent values 0..max_value
  int b = 1;
  while (b < 64 && (max_value >> b)) ++b;
  return b;
}
}  // namespace

// ------------------------------------------------------------------ small kernels
namespace sb {

__global__ void k_reset_step(Counters *c) {
  c->n_anchors = 0;
  c->n_hits = 0;
  c->n_queries = 0;
  c->n_capped = 0;
  c->n_events_raw = 0;
  c->n_events_kept = 0;
  c->n_linked = 0;
  c->n_pending = 0;
  c->n_segments = 0;
  c->work = 0;
  c->work2 = 0;
  c->n_overflow = 0;
  c->abort = 0;
  c->need_chain = 0;
  c->need_anchor = 0;
  c->sort_cursor = 0;
  c->n_cand = 0;
  c->max_entry_anchors = 0;
  c->dp_cursor = 0;
  c->error &= ~(24u | 64u);  // per-step bits (run table overflow, dense entry, query buffers); the others are per round
}

// queries per entry (spatial_index.cc:349-409 with Q3: seeds at step, 2*step, ... while
// count < (F-5)/step  =>  floor((F-6)/step) of them) and their exclusive scan; one block.
__global__ void k_query_table(const uint32_t *__restrict__ n_features, uint32_t B, uint32_t B_present,
                              int step, uint32_t *__restrict__ n_queries, uint32_t *__restrict__ q_off,
                              Counters *ctr) {
  __shared__ uint32_t warp_excl[32];
  __shared__ uint32_t tile_total;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  uint32_t carry = 0;  // identical in every thread
  for (uint32_t base = 0; base < B; base += blockDim.x) {
    const uint32_t b = base + threadIdx.x;
    uint32_t nq = 0;
    if (b < B_present) {
      const uint32_t F = n_features[b];
      if (F > (uint32_t)kMinFeatures) nq = (F - kDim) / (uint32_t)step;
    }
    uint32_t incl = nq;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    if (lane == 31) warp_excl[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      const uint32_t v = lane < n_warps ? warp_excl[lane] : 0;
      uint32_t in = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, in, d);
        if (lane >= d) in += t;
      }
      warp_excl[lane] = in - v;
      if (lane == 31) tile_total = in;
    }
    __syncthreads();
    if (b < B) {
      n_queries[b] = nq;
      q_off[b] = carry + warp_excl[wid] + (incl - nq);
    }
    carry += tile_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    q_off[B] = carry;
    ctr->n_queries = carry;
  }
}

__global__ void k_clear_error_bits(Counters *c, unsigned int bits) { c->error &= ~bits; }

__global__ void k_gather_round(const SlotState *__restrict__ slots, const uint32_t *__restrict__ ids,
                               uint32_t n, RoundInfo *__restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const SlotState &s = slots[ids[i]];
  out[i] = RoundInfo{s.stop, s.num_events, s.n_chains};
}

// stage hook: scatter user features (concatenated) into the [B][kFeatCap] layout
__global__ void k_scatter_features(const float *__restrict__ src, const uint32_t *__restrict__ feat_off,
                                   uint32_t B, float *__restrict__ dst, uint32_t *__restrict__ n_features) {
  const uint32_t b = blockIdx.x;
  if (b >= B) return;
  const uint32_t o = feat_off[b], n = min(feat_off[b + 1] - o, (uint32_t)kFeatCap);
  if (threadIdx.x == 0) n_features[b] = n;
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x)
    dst[(size_t)b * kFeatCap + i] = src[o + i];
}

// cached features: n_features of this step's entries from the lookahead block's rows (+ the
// event counters the events kernel would have bumped had it run inside this step)
__global__ void k_gather_nfeat(const uint32_t *__restrict__ nf_cache, const uint32_t *__restrict__ nraw_cache,
                               const uint32_t *__restrict__ feat_row, uint32_t B,
                               uint32_t *__restrict__ n_features, Counters *ctr) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t nf = 0, nr = 0;
  if (b < B) {
    const uint32_t row = feat_row[b];
    nf = nf_cache[row];
    nr = nraw_cache[row];
    n_features[b] = nf;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    nf += __shfl_xor_sync(0xffffffffu, nf, d);
    nr += __shfl_xor_sync(0xffffffffu, nr, d);
  }
  if ((threadIdx.x & 31) == 0 && (nf | nr)) {
    atomicAdd(&ctr->n_events_kept, (unsigned long long)nf);
    atomicAdd(&ctr->n_events_raw, (unsigned long long)nr);
  }
}

// stage hook: per-query hit counts from sorted (qid << 32 | widx) keys
__global__ void k_count_by_query(const uint64_t *__restrict__ key, unsigned long long n,
                                 unsigned long long *__restrict__ counts) {
  unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(&counts[key[i] >> 32], 1ull);
}

}  // namespace sb

struct smb_batch {
  smb_ctx *ctx;
  SlotSpace sp;
};

// persistent grid of the general search kernel: every CTA that fits on the device, no more
static size_t search_smem(const smb_ctx *ctx) { return kSearchWarps * search_smem_per_warp(ctx->index.ix.n_levels); }

template <bool STAGE>
static unsigned search_grid(smb_ctx *ctx) {
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_radius_search<STAGE>, kSearchWarps * 32,
                                                    search_smem(ctx)) != cudaSuccess || n < 1)
    n = 4;
  return ctx->n_sm * (unsigned)n;
}

void index_installed(smb_ctx *ctx) {
  ctx->search_grid_main = search_grid<false>(ctx);
  ctx->has_index = true;
}

// The whole radius search of one batch on stream s: Morton keys of the queries -> radix sort ->
// lean kernel over the sorted queries -> general kernel over the queries the lean one left.
// `sa` arrives with everything but the order / overflow fields filled in; nq_max bounds the
// number of queries (the exact count is only known on the device in pipeline mode).
template <bool STAGE>
static int launch_search(smb_ctx *ctx, SearchArgs sa, uint32_t nq_max, cudaStream_t s) {
  sa.nq_cap = nq_max;
  Workspace &w = ctx->ws;
  const size_t gsm = search_smem(ctx);
  if (!ctx->search_lean || nq_max == 0) {
    sa.work = &ctx->d_ctr.p->work;
    k_radius_search<STAGE><<<STAGE ? search_grid<true>(ctx) : ctx->search_grid_main, kSearchWarps * 32, gsm, s>>>(ctx->index.ix, sa);
    LAUNCH_CHECK();
    return SMB_OK;
  }
  CK(w.ovf_list.ensure(nq_max));
  if (!STAGE) CK(w.entry_info.ensure(sa.B));
  if (nq_max < ctx->sort_queries_min) {
    // a small batch (a read-until round) fits the caches whatever the order: the queries keep their
    // natural order (consecutive queries share an entry, so a flush serves several of them) and the
    // round saves the key kernel and the five launches of the radix sort
    if (!STAGE) {
      k_entry_info<<<(sa.B + 255) / 256, 256, 0, s>>>(sa.feat_row, sa.entry_slot, sa.slots, sa.B, w.entry_info.p);
      LAUNCH_CHECK();
    }
    sa.order = nullptr;
    sa.nq_cap = 0xFFFFFFFFu;
  } else {
    CK(w.qkey_a.ensure(nq_max));
    CK(w.qkey_b.ensure(nq_max));
    CK(w.qpay_a.ensure(nq_max));
    CK(w.qpay_b.ensure(nq_max));
    if (STAGE) {
      k_query_keys_stage<<<(nq_max + 255) / 256, 256, 0, s>>>(sa.features, nq_max, ctx->index.ix.vmin, ctx->index.ix.inv_span,
                                                              w.qkey_a.p, w.qpay_a.p);
    } else {
      // entries without queries write nothing; the sort only looks at the first q_off[B] keys,
      // but it is sized on the host: pad the tail with the largest key so it stays at the end
      CK(cudaMemsetAsync(w.qkey_a.p, 0xFF, (size_t)nq_max * sizeof(uint32_t), s));
      k_query_keys<<<sa.B, 128, 0, s>>>(sa.features, sa.feat_row, sa.q_off, sa.entry_slot, sa.slots, sa.B, sa.step,
                                        ctx->index.ix.vmin, ctx->index.ix.inv_span, w.qkey_a.p, w.qpay_a.p, w.entry_info.p, nq_max);
    }
    LAUNCH_CHECK();
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, w.qkey_a.p, w.qkey_b.p, w.qpay_a.p, w.qpay_b.p, (int)nq_max, 0, 24, s);
    CK(w.qsort_temp.ensure(tb));
    CK(cub::DeviceRadixSort::SortPairs(w.qsort_temp.p, tb, w.qkey_a.p, w.qkey_b.p, w.qpay_a.p, w.qpay_b.p, (int)nq_max,
                                       0, 24, s));
    ctx->stats.launches += 5;
    sa.order = w.qpay_b.p;
  }
  sa.stage_cap = lean_stage_cap(ctx->index.ix.smem_bytes);
  sa.entry_info = w.entry_info.p;
  sa.front_cap = std::min<uint32_t>(std::max<uint32_t>(ctx->front_cap, 72u), (uint32_t)kFrontCap);
  sa.ovf_list = w.ovf_list.p;
  sa.work = &ctx->d_ctr.p->work;
  k_search_lean<STAGE><<<ctx->n_sm, kLeanWarps * 32, lean_smem(ctx->index.ix.smem_bytes, sa.stage_cap), s>>>(ctx->index.ix, sa);
  LAUNCH_CHECK();
  // the queries whose frontier outgrew the lean kernel's slots (none, mostly: the launch then
  // finds an empty list and returns)
  sa.qlist = w.ovf_list.p;
  sa.qlist_n = &ctx->d_ctr.p->n_overflow;
  sa.work = &ctx->d_ctr.p->work2;
  k_radius_search<STAGE><<<STAGE ? search_grid<true>(ctx) : ctx->search_grid_main, kSearchWarps * 32, gsm, s>>>(ctx->index.ix, sa);
  LAUNCH_CHECK();
  return SMB_OK;
}

// ------------------------------------------------------------------ the pipeline step
enum StepSource { SRC_RAW_KEPT, SRC_PA_FLOAT, SRC_FEATURES, SRC_CACHED };

struct StepEntries {
  uint32_t B = 0, B_present = 0;           // present entries first, absent ones after
  std::vector<uint32_t> slot;
  std::vector<uint64_t> chunk_start;       // SRC_RAW_KEPT / SRC_PA_FLOAT: sample index of the chunk
  std::vector<float> offset, scale;        // SRC_RAW_KEPT
  const void *samples = nullptr;           // device pointer (kept int16 or pA float)
  const float *d_features = nullptr;       // SRC_FEATURES: concatenated features (device)
  const uint32_t *d_feat_off = nullptr;    // SRC_FEATURES: B_present+1 offsets (device)
  std::vector<uint32_t> feat_row;          // SRC_CACHED: row of each present entry in ws.feat_cache
};

static int ensure_event_ws(smb_ctx *ctx, uint32_t B) {
  Workspace &w = ctx->ws;
  const uint32_t Bp = (B + 31) & ~31u;
  const size_t tr = (size_t)(kChunk + 1) * Bp;
  CK(w.ps.ensure(tr));
  CK(w.pss.ensure(tr));
  CK(w.t1.ensure(tr));
  CK(w.t2.ensure(tr));
  CK(w.means.ensure((size_t)B * kFeatCap));
  return SMB_OK;
}

struct ChunkTable {  // device arrays describing the chunks of one event launch
  const uint64_t *start;
  const float *offset, *scale;
};

static int run_events(smb_ctx *ctx, StepSource src, const void *samples, uint32_t B,
                      uint32_t *d_peaks_out, float *d_features = nullptr, uint32_t *d_n_features = nullptr,
                      uint32_t *d_n_raw = nullptr, cudaStream_t s = nullptr, const ChunkTable *table = nullptr) {
  Workspace &w = ctx->ws;
  if (!s) s = ctx->stream;
  const ChunkTable own{w.chunk_start.p, w.chunk_offset.p, w.chunk_scale.p};
  const ChunkTable &ct = table ? *table : own;
  const uint32_t Bp = (B + 31) & ~31u;
  // small batches (read-until rounds, the thin last rounds of a read set): a warp per chunk in
  // shared memory; the stage hook that returns the t-statistics needs the global arrays
  if (B <= ctx->ev_warp_max && !d_peaks_out) {
    CK(w.means.ensure((size_t)B * kFeatCap));
    if (!d_n_raw) CK(w.n_raw_events.ensure(B));
    float *feat = d_features ? d_features : w.features.p;
    uint32_t *nfeat = d_n_features ? d_n_features : w.n_features.p;
    uint32_t *nraw = d_n_raw ? d_n_raw : w.n_raw_events.p;
    Counters *ctr = d_n_raw ? nullptr : ctx->d_ctr.p;
    if (src == SRC_RAW_KEPT)
      k_ev_chunk_warp<true><<<B, 32, kEvWarpSmem, s>>>(samples, ct.start, ct.offset, ct.scale,
                                                       w.means.p, feat, nfeat, nraw, nullptr, B, ctr);
    else
      k_ev_chunk_warp<false><<<B, 32, kEvWarpSmem, s>>>(samples, ct.start, nullptr, nullptr, w.means.p,
                                                        feat, nfeat, nraw, nullptr, B, ctr);
    LAUNCH_CHECK();
    return SMB_OK;
  }
  int rc = ensure_event_ws(ctx, B);
  if (rc) return rc;
  if (src == SRC_RAW_KEPT)
    k_ev_prefix<true><<<(B + 127) / 128, 128, 0, s>>>(samples, ct.start, ct.offset, ct.scale, w.ps.p, w.pss.p,
                                                      B, Bp);
  else
    k_ev_prefix<false><<<(B + 127) / 128, 128, 0, s>>>(samples, ct.start, nullptr, nullptr,
                                                       w.ps.p, w.pss.p, B, Bp);
  LAUNCH_CHECK();
  dim3 g((B + 127) / 128, (kChunk + 1 + kStrip - 1) / kStrip);
  k_ev_tstat<<<g, 128, 0, s>>>(w.ps.p, w.pss.p, w.t1.p, w.t2.p, B, Bp);
  LAUNCH_CHECK();
  if (!d_n_raw) CK(w.n_raw_events.ensure(B));
  k_ev_features<<<(B + 127) / 128, 128, 0, s>>>(w.t1.p, w.t2.p, w.ps.p, w.means.p,
                                                d_features ? d_features : w.features.p,
                                                d_n_features ? d_n_features : w.n_features.p,
                                                d_n_raw ? d_n_raw : w.n_raw_events.p, d_peaks_out, B, Bp,
                                                d_n_raw ? nullptr : ctx->d_ctr.p);
  LAUNCH_CHECK();
  return SMB_OK;
}

// How a step's anchors get sorted; a path that cannot take the step (run tables overflowed, a part
// or an entry too dense for shared memory) aborts it on the device and the host redoes the step
// one path down.
enum SortMode { SORT_PART = 0, SORT_SEG = 1, SORT_GLOBAL = 2 };

// what the end of a round wants read back together with the last step's counters
struct RoundOut {
  const std::vector<uint32_t> *ids = nullptr;  // slots whose (stop, events, chains) go to info
  std::vector<RoundInfo> *info = nullptr;
  std::vector<SlotState> *states = nullptr;    // all slots of the space, when asked for
};

static int host_sync(smb_ctx *ctx) {
  ctx->stats.sync_points++;
  CK(cudaStreamSynchronize(ctx->stream));
  return SMB_OK;
}

namespace sb {
// after the search: everything the host used to decide from the counters, decided here
__global__ void k_step_check(Counters *c, unsigned long long cap, int sort_mode, unsigned int part_limit,
                             unsigned long long seg_limit, uint32_t n_parts) {
  unsigned int ab = 0;
  if (c->n_anchors > cap) ab |= kAbortAnchors;
  if (c->error & 64u) ab |= kAbortQueries;
  if (sort_mode == 0 && ((c->error & 8u) || c->max_entry_anchors > part_limit)) ab |= kAbortSort;
  if (sort_mode == 1 && ((c->error & 8u) || (unsigned long long)c->max_entry_anchors * n_parts > seg_limit)) ab |= kAbortSort;
  c->abort |= ab;
}
// global-sort path: keys past the step's anchors must sort to the end (the radix sort is sized
// for the buffers on the host)
__global__ void k_pad_keys(uint64_t *__restrict__ key, const Counters *__restrict__ c, unsigned long long cap) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < cap && i >= c->n_anchors) key[i] = ~0ull;
}
}  // namespace sb

// grow a carry pool without losing what the earlier steps of the round put there
template <class T>
static cudaError_t grow_keep(DevBuf<T> &buf, size_t want, cudaStream_t s) {
  if (want <= buf.cap) return cudaSuccess;
  DevBuf<T> bigger;
  cudaError_t e = bigger.ensure(want);
  if (e != cudaSuccess) return e;
  if (buf.p && buf.cap) {
    e = cudaMemcpyAsync(bigger.p, buf.p, buf.cap * sizeof(T), cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return e;
  }
  buf = std::move(bigger);
  return cudaSuccess;
}

// One pipeline step, enqueued without a host round trip; the host looks at the counters once, at
// the end.  Returns SMB_OK, an error, +1 when the anchor buffers overflowed (the caller grows them
// or splits the batch), +2 when the step was aborted for another reason that has been dealt with
// (estimates raised, pools grown, *sort_mode moved one path down): the caller just runs it again.
// Nothing is committed to the read slots by an aborted step.
static int run_step(smb_ctx *ctx, SlotSpace &sp, const StepEntries &en, StepSource src,
                    const smb_params &prm, uint32_t out_pool, int *sort_mode, const RoundOut *rout) {
  Workspace &w = ctx->ws;
  cudaStream_t s = ctx->stream;
  const uint32_t B = en.B, Bpres = en.B_present;
  if (B == 0) return SMB_OK;
  if (!ctx->has_index) return fail(ctx, SMB_ERR_STATE, "no index loaded");
  const bool sharded = ctx->ex && ctx->index.sharded;
  // ---- key layout for this step
  uint32_t max_ev = 0;
  for (uint32_t b = 0; b < Bpres; ++b) max_ev = std::max(max_ev, sp.h_events[en.slot[b]]);
  KeyLayout kl;
  kl.qbits = bits_for((uint64_t)max_ev + kFeatCap);
  kl.tbits = bits_for(ctx->index.max_tpos);
  kl.bbits = bits_for(ctx->index.max_bucket);
  kl.ebits = bits_for(B - 1);
  if (kl.total() > 64) return fail(ctx, SMB_ERR_CAPACITY, "sort key exceeds 64 bits: lower max_batch_chunks");
  if (ctx->max_batch_anchors >= (1ull << 30)) return fail(ctx, SMB_ERR_ARG, "max_batch_anchors must stay below 2^30");
  // anchor buffers sized from the running estimate (they grow on overflow, up to the limit)
  // (the step's capacity follows the estimate, not the buffers' high-water mark: grids that are
  // sized for it -- k_chain_prep -- would otherwise launch mostly empty blocks on small steps)
  const uint64_t cap = std::min<uint64_t>(
      ctx->max_batch_anchors, (uint64_t)(1.5 * ctx->est_anchors_per_chunk * std::max(Bpres, 1u)) + (1u << 20));
  ctx->last_cap = cap;

  // ---- per-entry arrays
  CK(w.entry_slot.ensure(B));
  CK(w.absent.ensure(B));
  CK(w.n_features.ensure(B));
  CK(w.n_raw_events.ensure(B));
  CK(w.n_queries.ensure(B));
  CK(w.q_off.ensure(B + 1));
  if (src != SRC_CACHED) CK(w.features.ensure((size_t)std::max(Bpres, 1u) * kFeatCap));
  CK(w.feat_row.ensure(B));
  CK(cudaMemcpyAsync(w.entry_slot.p, en.slot.data(), B * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
  ctx->stats.h2d_bytes += B * sizeof(uint32_t);
  {
    // feature row of every entry: identity into ws.features, or rows of the lookahead block
    std::vector<uint32_t> &rows = ctx->h_feat_row;
    rows.resize(B);
    for (uint32_t b = 0; b < B; ++b) rows[b] = (src == SRC_CACHED && b < Bpres) ? en.feat_row[b] : (b < Bpres ? b : 0);
    CK(cudaMemcpyAsync(w.feat_row.p, rows.data(), B * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += B * sizeof(uint32_t);
  }
  CK(cudaEventRecord(ctx->ev[0], s));
  k_reset_step<<<1, 1, 0, s>>>(ctx->d_ctr.p);
  LAUNCH_CHECK();
  CK(cudaMemsetAsync(w.n_features.p, 0, B * sizeof(uint32_t), s));
  if (Bpres > 0) {
    if (src == SRC_FEATURES) {
      k_scatter_features<<<Bpres, 256, 0, s>>>(en.d_features, en.d_feat_off, Bpres, w.features.p, w.n_features.p);
      LAUNCH_CHECK();
    } else if (src == SRC_CACHED) {
      k_gather_nfeat<<<(Bpres + 255) / 256, 256, 0, s>>>(w.nf_cache[w.cache_cur].p, w.nraw_cache[w.cache_cur].p, w.feat_row.p, Bpres,
                                                         w.n_features.p, ctx->d_ctr.p);
      LAUNCH_CHECK();
    } else {
      CK(w.chunk_start.ensure(Bpres));
      CK(cudaMemcpyAsync(w.chunk_start.p, en.chunk_start.data(), Bpres * sizeof(uint64_t),
                         cudaMemcpyHostToDevice, s));
      ctx->stats.h2d_bytes += Bpres * sizeof(uint64_t);
      if (src == SRC_RAW_KEPT) {
        CK(w.chunk_offset.ensure(Bpres));
        CK(w.chunk_scale.ensure(Bpres));
        CK(cudaMemcpyAsync(w.chunk_offset.p, en.offset.data(), Bpres * sizeof(float), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(w.chunk_scale.p, en.scale.data(), Bpres * sizeof(float), cudaMemcpyHostToDevice, s));
        ctx->stats.h2d_bytes += 2 * Bpres * sizeof(float);
      }
      int rc = run_events(ctx, src, en.samples, Bpres, nullptr);
      if (rc) return rc;
    }
  }
  CK(cudaEventRecord(ctx->ev[1], s));
  k_query_table<<<1, 1024, 0, s>>>(w.n_features.p, B, Bpres, prm.step_size, w.n_queries.p, w.q_off.p, ctx->d_ctr.p);
  LAUNCH_CHECK();

  // ---- anchors: carried ones first, then the radius search appends its hits
  CK(w.key_a.ensure(cap));
  CK(w.key_b.ensure(cap));
  CK(w.dist_a.ensure(cap));
  CK(w.dist_b.ensure(cap));
  CK(w.score.ensure(cap));
  CK(w.coef.ensure(cap));
  CK(w.pred.ensure(cap));
  int mode = std::max(*sort_mode, !ctx->seg_sort ? (int)SORT_GLOBAL : (!ctx->part_sort ? (int)SORT_SEG : (int)SORT_PART));
  const bool want_seg = mode != SORT_GLOBAL;
  // parts per entry (k_sort.cuh): equal coordinate ranges sized so that a part of an average
  // entry fills kPartFill (70 %) of one k_part_sort CTA; more than kMaxParts -> one list, k_seg_sort
  constexpr double kPartFill = 0.70;
  uint32_t n_parts = 1;
  uint64_t span = std::max<uint64_t>(ctx->index.g_total, 1);
  if (mode == SORT_PART) {
    const double per_coord = std::max(ctx->est_anchors_per_chunk, 1.0) / (double)std::max<uint64_t>(ctx->index.g_total, 1);
    const double want = kPartFill * (double)kPartSortCap / per_coord;
    if (want < (double)ctx->index.g_total) {
      const uint64_t sp2 = std::max<uint64_t>((uint64_t)want, 1);
      const uint64_t np = (ctx->index.g_total + sp2 - 1) / sp2;
      if (np <= (uint64_t)kMaxParts) {
        n_parts = (uint32_t)np;
        span = sp2;
      }
    }
  }
  const float inv_span = 1.0f / (float)span;
  const size_t n_lists = (size_t)B * n_parts;
  // run records per (entry, part) list: a query leaves at most one run per part and flush, so
  // queries per chunk + the flushes forced by a full staging buffer, with room for dense chunks
  uint32_t runs_cap = (uint32_t)(ctx->runs_scale * (1.5 * ctx->est_queries_per_chunk +
                                                    3.0 * ctx->est_anchors_per_chunk / (double)kStageCap)) + 128u;
  runs_cap = (runs_cap + 63u) & ~63u;
  if (ctx->runs_cap_min) runs_cap = ctx->runs_cap_min;
  if (want_seg) {
    CK(w.runs.ensure(n_lists * runs_cap));
    CK(w.run_count.ensure(n_lists));
    CK(w.entry_total.ensure(n_lists));
    CK(w.part_base.ensure(n_lists + 1));
    CK(cudaMemsetAsync(w.run_count.p, 0, n_lists * sizeof(uint32_t), s));
    CK(cudaMemsetAsync(w.entry_total.p, 0, n_lists * sizeof(uint32_t), s));
  }
  const uint64_t n_slots64 = (uint64_t)B << kl.bbits;
  if (n_slots64 >= (1ull << 31)) return fail(ctx, SMB_ERR_CAPACITY, "segment table too large: lower max_batch_chunks");
  CK(w.seg_qmin.ensure((size_t)n_slots64));
  k_seg_qmin_init<<<(unsigned)((n_slots64 + 255) / 256), 256, 0, s>>>(w.entry_slot.p, sp.slots.p, (uint32_t)n_slots64,
                                                                       kl.bbits, w.seg_qmin.p);
  LAUNCH_CHECK();
  k_inject_carry<<<(B * 32 + kCarryThreads - 1) / kCarryThreads, kCarryThreads, 0, s>>>(
      w.entry_slot.p, w.n_queries.p, sp.slots.p, sp.pool_anchor[0].p, sp.pool_anchor[1].p, B, kl, w.key_a.p,
      w.dist_a.p, cap, ctx->d_ctr.p, want_seg ? w.runs.p : nullptr, w.run_count.p, w.entry_total.p,
      runs_cap, n_parts, inv_span, ctx->index.bucket_base.p, w.seg_qmin.p);
  LAUNCH_CHECK();
  SearchArgs sa{};
  sa.features = src == SRC_CACHED ? w.feat_cache[w.cache_cur].p : w.features.p;
  sa.feat_row = w.feat_row.p;
  sa.q_off = w.q_off.p;
  sa.entry_slot = w.entry_slot.p;
  sa.slots = sp.slots.p;
  sa.slots_mut = sp.slots.p;
  sa.B = B;
  sa.step = prm.step_size;
  sa.radius = prm.search_radius;
  sa.key = kl;
  sa.out_key = w.key_a.p;
  sa.out_dist = w.dist_a.p;
  sa.cap = cap;
  sa.ctr = ctx->d_ctr.p;
  sa.runs = want_seg ? w.runs.p : nullptr;
  sa.run_count = w.run_count.p;
  sa.entry_total = w.entry_total.p;
  sa.runs_cap = runs_cap;
  sa.n_parts = n_parts;
  sa.inv_span = inv_span;
  sa.bucket_base = ctx->index.bucket_base.p;
  sa.n_buckets = ctx->index.max_bucket + 1u;
  // query-order buffers are sized from a running estimate (the exact count is on the device)
  const uint32_t q_per_chunk_max = (uint32_t)(kFeatCap - kDim) / (uint32_t)prm.step_size;
  const uint32_t nq_max = (uint32_t)std::min<uint64_t>(
      (uint64_t)Bpres * q_per_chunk_max, (uint64_t)(1.25 * ctx->est_queries_per_chunk * Bpres) + 4096u);
  CK(cudaEventRecord(ctx->ev[2], s));
  {
    int rc = launch_search<false>(ctx, sa, nq_max, s);
    if (rc) return rc;
  }
  ctx->stats.search_launches++;
  CK(cudaEventRecord(ctx->ev[3], s));
  if (want_seg) {
    k_max_u32<<<148, 256, 0, s>>>(w.entry_total.p, n_lists, &ctx->d_ctr.p->max_entry_anchors);
    LAUNCH_CHECK();
  }
  if (sharded) {
    // Sharded: every rank must take the same path through this step (the exchanges below are
    // collective), so overflow and the estimate are agreed on first -- with a host round trip.
    CK(cudaMemcpyAsync(ctx->h_ctr.p, ctx->d_ctr.p, sizeof(Counters), cudaMemcpyDeviceToHost, s));
    int rc = host_sync(ctx);
    if (rc) return rc;
    ctx->stats.d2h_bytes += sizeof(Counters);
    const unsigned long long n_local = ctx->h_ctr.p->n_anchors;
    const bool overflow_local = n_local > cap;
    CK(w.ctl.ensure(4));
    ctx->h_ctl.p[0] = overflow_local ? 1.0 : 0.0;
    ctx->h_ctl.p[1] = (overflow_local && ctx->last_cap >= ctx->max_batch_anchors) ? 1.0 : 0.0;
    ctx->h_ctl.p[2] = (double)n_local;
    ctx->h_ctl.p[3] = (ctx->h_ctr.p->error & 64u) ? 1.0 : 0.0;
    CK(cudaMemcpyAsync(w.ctl.p, ctx->h_ctl.p, 4 * sizeof(double), cudaMemcpyHostToDevice, s));
    rc = ctx->ex->allreduce(w.ctl.p, 4, EX_F64, EX_MAX, s, ctx->err);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->h_ctl.p, w.ctl.p, 4 * sizeof(double), cudaMemcpyDeviceToHost, s));
    rc = host_sync(ctx);
    if (rc) return rc;
    ctx->stats.exchanges++;
    ctx->group_at_limit = ctx->h_ctl.p[1] > 0.0;
    if (ctx->h_ctl.p[3] > 0.0) {  // some rank ran out of query-order slots: everybody redoes the step
      ctx->est_queries_per_chunk = 1.1 * (double)q_per_chunk_max;
      return 2;
    }
    if (ctx->h_ctl.p[0] > 0.0) return 1;  // nothing has been committed to the slots yet
  }
  k_step_check<<<1, 1, 0, s>>>(ctx->d_ctr.p, cap, mode, 8u * (unsigned)kPartSortCap, 8ull * (unsigned)kSortCapBig, n_parts);
  LAUNCH_CHECK();

  // ---- sort by (entry, bucket, target, query)
  CK(cudaEventRecord(ctx->ev[4], s));
  const uint64_t *keys = w.key_b.p;
  const float *dists = w.dist_b.p;
  if (mode == SORT_PART) {
    // one CTA per (entry, part) from the pre-routed runs; output offsets = scan of the part sizes
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, w.entry_total.p, w.part_base.p, (int)n_lists, s);
    CK(w.cub_temp.ensure(tb));
    CK(cub::DeviceScan::ExclusiveSum(w.cub_temp.p, tb, w.entry_total.p, w.part_base.p, (int)n_lists, s));
    ctx->stats.launches += 2;
    PartSortArgs ps{};
    ps.key_in = w.key_a.p;
    ps.dist_in = w.dist_a.p;
    ps.key_out = w.key_b.p;
    ps.dist_out = w.dist_b.p;
    ps.runs = w.runs.p;
    ps.run_count = w.run_count.p;
    ps.runs_cap = runs_cap;
    ps.part_total = w.entry_total.p;
    ps.out_base = w.part_base.p;
    ps.n_parts = n_parts;
    ps.span = span;
    ps.kl = kl;
    ps.bucket_base = ctx->index.bucket_base.p;
    ps.n_buckets = ctx->index.max_bucket + 1u;
    ps.ctr = ctx->d_ctr.p;
    k_part_sort<kPartSortCap, 512, 4096><<<(unsigned)n_lists, 512, part_sort_smem_bytes(kPartSortCap, 4096), s>>>(ps);
    LAUNCH_CHECK();
  } else if (mode == SORT_SEG) {
    // one CTA per entry working through the entry in several passes
    SegSortArgs ss{};
    ss.key_in = w.key_a.p;
    ss.dist_in = w.dist_a.p;
    ss.key_out = w.key_b.p;
    ss.dist_out = w.dist_b.p;
    ss.runs = w.runs.p;
    ss.run_count = w.run_count.p;
    ss.runs_cap = runs_cap;
    ss.n_parts = n_parts;
    ss.B = B;
    ss.kl = kl;
    ss.bucket_base = ctx->index.bucket_base.p;
    ss.gshift = ctx->index.gshift;
    ss.n_coarse = ctx->index.n_coarse;
    ss.ctr = ctx->d_ctr.p;
    k_seg_sort<kSortCapBig, 1024, 8192><<<B, 1024, sort_smem_bytes(kSortCapBig, 8192), s>>>(ss);
    LAUNCH_CHECK();
  } else {
    // radix sort on (entry, bucket, target) only; k_fix_ties orders equal-target runs by query.
    // The sort is sized for the buffers (the count lives on the device): the slots past the
    // step's anchors are filled with the largest key and stay at the end.
    k_pad_keys<<<(unsigned)((cap + 255) / 256), 256, 0, s>>>(w.key_a.p, ctx->d_ctr.p, cap);
    LAUNCH_CHECK();
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, w.key_a.p, w.key_b.p, w.dist_a.p, w.dist_b.p,
                                    (uint64_t)cap, kl.qbits, 64, s);
    CK(w.cub_temp.ensure(tb));
    CK(cub::DeviceRadixSort::SortPairs(w.cub_temp.p, tb, w.key_a.p, w.key_b.p, w.dist_a.p, w.dist_b.p,
                                       (uint64_t)cap, kl.qbits, 64, s));
    ctx->stats.launches += 2 + (64 - kl.qbits + 7) / 8;
    k_fix_ties<<<(unsigned)((cap + 255) / 256), 256, 0, s>>>(w.key_b.p, w.dist_b.p, ctx->d_ctr.p, kl.qbits);
    LAUNCH_CHECK();
  }
  CK(cudaEventRecord(ctx->ev[5], s));

  // ---- chaining
  ChainArgs ca{};
  ca.key = keys;
  ca.dist = dists;
  ca.n_max = cap;
  ca.kl = kl;
  ca.radius = prm.search_radius;
  ca.score = w.score.p;
  ca.coef = w.coef.p;
  ca.pred = w.pred.p;
  ca.n_slots = (uint32_t)n_slots64;
  ca.seg_qmin = w.seg_qmin.p;
  CK(w.seg.ensure(ca.n_slots));
  CK(w.seg_max.ensure(ca.n_slots));
  ca.seg = w.seg.p;
  ca.seg_max = w.seg_max.p;
  ca.ctr = ctx->d_ctr.p;
  ca.dp_passes = ctx->dp_passes;
  CK(cudaMemsetAsync(w.seg.p, 0xFF, (size_t)ca.n_slots * sizeof(SegRec), s));
  CK(cudaMemsetAsync(w.seg_max.p, 0, (size_t)ca.n_slots * sizeof(float), s));
  const unsigned n_tiles = (unsigned)((cap + kPrepTile - 1) / kPrepTile);  // sized for the buffers
  CK(w.link_list.ensure((size_t)std::max(n_tiles, 1u) * kPrepTile));
  CK(w.link_count.ensure(std::max(n_tiles, 1u)));
  CK(w.pend_list.ensure((size_t)std::max(n_tiles, 1u) * kPrepTile));
  CK(w.pend_count.ensure(std::max(n_tiles, 1u)));
  ca.link_list = w.link_list.p;
  ca.link_count = w.link_count.p;
  ca.pend_list = w.pend_list.p;
  ca.pend_count = w.pend_count.p;
  ca.prep_rounds = ctx->prep_rounds;
  k_chain_prep<<<n_tiles, kPrepThreads, 0, s>>>(ca);
  LAUNCH_CHECK();
  if (B <= ctx->dp_pass_max_entries) {  // small batch: per-tile parallel pass first (latency)
    k_dp_pass<<<ctx->n_sm * 6u, kDpPassThreads, 0, s>>>(ca);
    LAUNCH_CHECK();
  }
  {
    const unsigned dp_blocks = (unsigned)(((uint64_t)ca.n_slots * 32 + kDpThreads - 1) / kDpThreads);
    k_chain_dp<<<std::min(dp_blocks, ctx->dp_grid), kDpThreads, 0, s>>>(ca);
    LAUNCH_CHECK();
  }
  SelectArgs se{};
  se.c = ca;
  se.entry_slot = w.entry_slot.p;
  se.n_queries = w.n_queries.p;
  se.n_features = w.n_features.p;
  se.slots = sp.slots.p;
  se.B = B;
  se.max_chains = std::min<uint32_t>(3u * (ctx->index.max_bucket + 1u), 4096u);
  CK(w.chain_tmp.ensure((size_t)B * se.max_chains));
  CK(w.n_scratch.ensure(B));
  CK(w.pick.ensure(B));
  se.scratch = w.chain_tmp.p;
  se.n_scratch = w.n_scratch.p;
  se.path = w.link_list.p;  // the DP is done with its work lists: reuse them for the chain paths
  se.rank = sharded ? (uint32_t)ctx->ex->rank : 0u;
  se.out_pool = out_pool;
  for (int p = 0; p < 2; ++p) {
    se.pool_chain[p] = sp.pool_chain[p].p;
    se.pool_anchor[p] = sp.pool_anchor[p].p;
  }
  se.pool_chain_cap = sp.pool_chain[out_pool].cap;
  se.pool_anchor_cap = sp.pool_anchor[out_pool].cap;
  se.prm = prm;
  CK(cudaMemsetAsync(w.n_scratch.p, 0, B * sizeof(uint32_t), s));
  if (sharded) {
    // exchange 2: the per-bucket running max of every rank's own contigs
    int rc = ctx->ex->allreduce(w.seg_max.p, ca.n_slots, EX_F32, EX_MAX, s, ctx->err);
    if (rc) return rc;
    // a chain has >= 2 anchors of its own and a segment yields <= 3 of them
    se.cand_cap = (uint32_t)std::min<uint64_t>(3ull * ca.n_slots, cap / 2) + 1u;
    CK(w.cand_list.ensure(se.cand_cap));
    se.cand_list = w.cand_list.p;
    ctx->stats.exchanges++;
  }
  k_sel_trace<<<(unsigned)(((uint64_t)ca.n_slots * 32 + kTraceThreads - 1) / kTraceThreads), kTraceThreads, 0, s>>>(se);
  LAUNCH_CHECK();
  if (sharded) {
    // exchange 3: candidate counts, then the candidate records padded to the largest count
    const uint32_t world = (uint32_t)ctx->ex->world;
    CK(w.cand_counts.ensure(world + 1));
    int rc = ctx->ex->allgather(&ctx->d_ctr.p->n_cand, w.cand_counts.p, sizeof(unsigned long long), s, ctx->err);
    if (rc) return rc;
    std::vector<unsigned long long> h_counts(world);
    CK(cudaMemcpyAsync(h_counts.data(), w.cand_counts.p, world * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    rc = host_sync(ctx);
    if (rc) return rc;
    unsigned long long per_rank = 0;
    for (uint32_t r = 0; r < world; ++r) per_rank = std::max(per_rank, h_counts[r]);
    if (per_rank > 0) {
      // my own list must be able to serve a padded send of per_rank records
      if (w.cand_list.cap < per_rank) {
        cudaError_t ge = grow_keep(w.cand_list, (size_t)per_rank, s);
        if (ge != cudaSuccess) return fail(ctx, SMB_ERR_CUDA, cudaGetErrorString(ge));
        se.cand_list = w.cand_list.p;
      }
      CK(w.cand_all.ensure((size_t)per_rank * world));
      rc = ctx->ex->allgather(w.cand_list.p, w.cand_all.p, (size_t)per_rank * sizeof(CandRec), s, ctx->err);
      if (rc) return rc;
      const uint64_t total = per_rank * world;
      k_sel_scatter<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(se, w.cand_all.p, w.cand_counts.p, world, (uint32_t)per_rank);
      LAUNCH_CHECK();
    }
    ctx->stats.exchanges += 2;
  }
  const unsigned final_blocks = (unsigned)(((uint64_t)B * 32 + kFinalThreads - 1) / kFinalThreads);
  k_sel_pick<<<final_blocks, kFinalThreads, 0, s>>>(se, w.pick.p);
  LAUNCH_CHECK();
  k_pool_check<<<1, 1, 0, s>>>(ctx->d_ctr.p, out_pool, se.pool_chain_cap, se.pool_anchor_cap);
  LAUNCH_CHECK();
  if (sharded) {
    // a rank-local abort (sort path, carry pools) becomes everybody's: all ranks redo the step
    int rc = ctx->ex->allreduce(&ctx->d_ctr.p->abort, 1, EX_U32, EX_MAX, s, ctx->err);
    if (rc) return rc;
    ctx->stats.exchanges++;
  }
  k_sel_commit<<<final_blocks, kFinalThreads, 0, s>>>(se, w.pick.p);
  LAUNCH_CHECK();
  CK(cudaEventRecord(ctx->ev[6], s));
  // ---- the step's one look at the device: counters, and what the round wants read back
  CK(cudaMemcpyAsync(ctx->h_ctr.p, ctx->d_ctr.p, sizeof(Counters), cudaMemcpyDeviceToHost, s));
  ctx->stats.d2h_bytes += sizeof(Counters);
  uint32_t n_ids = 0;
  if (rout && rout->ids && rout->info) {
    n_ids = (uint32_t)rout->ids->size();
    rout->info->resize(n_ids);
    if (n_ids) {
      CK(w.ids.ensure(n_ids));
      CK(w.round_info.ensure(n_ids));
      CK(cudaMemcpyAsync(w.ids.p, rout->ids->data(), n_ids * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
      k_gather_round<<<(n_ids + 255) / 256, 256, 0, s>>>(sp.slots.p, w.ids.p, n_ids, w.round_info.p);
      LAUNCH_CHECK();
      CK(cudaMemcpyAsync(rout->info->data(), w.round_info.p, n_ids * sizeof(RoundInfo), cudaMemcpyDeviceToHost, s));
      ctx->stats.h2d_bytes += n_ids * sizeof(uint32_t);
      ctx->stats.d2h_bytes += n_ids * sizeof(RoundInfo);
    }
  }
  if (rout && rout->states) {
    rout->states->resize(std::max<size_t>(sp.n_slots, 1));
    if (sp.n_slots) {
      CK(cudaMemcpyAsync(rout->states->data(), sp.slots.p, sp.n_slots * sizeof(SlotState), cudaMemcpyDeviceToHost, s));
      ctx->stats.d2h_bytes += sp.n_slots * sizeof(SlotState);
    }
  }
  {
    int rc = host_sync(ctx);
    if (rc) return rc;
  }
  const Counters &hc = *ctx->h_ctr.p;
  if (hc.abort) {
    // nothing was committed; adjust what was too small and let the caller run the step again
    if (hc.abort & kAbortAnchors) return 1;
    if (hc.abort & kAbortQueries)
      ctx->est_queries_per_chunk = 1.1 * (double)hc.n_queries / std::max(Bpres, 1u) + 8.0;
    if (hc.abort & kAbortSort) {
      if ((hc.error & 8u) && !ctx->runs_cap_min && ctx->runs_scale < 64.0) ctx->runs_scale *= 2.0;  // run tables overflowed
      else *sort_mode = mode + 1;                                        // a part / an entry too dense
      if (mode == SORT_GLOBAL) return fail(ctx, SMB_ERR_CAPACITY, "sort aborted on the radix path");
    }
    if (hc.abort & kAbortPool) {
      const size_t want_c = (size_t)(hc.carry_chain_used[out_pool] + hc.need_chain) * 2 + 64;
      const size_t want_a = (size_t)(hc.carry_anchor_used[out_pool] + hc.need_anchor) * 2 + 64;
      cudaError_t ge = grow_keep(sp.pool_chain[out_pool], want_c, s);
      if (ge == cudaSuccess) ge = grow_keep(sp.pool_anchor[out_pool], want_a, s);
      if (ge != cudaSuccess) return fail(ctx, SMB_ERR_CUDA, std::string("growing the carry pools: ") + cudaGetErrorString(ge));
    }
    return 2;
  }
  const unsigned long long n = hc.n_anchors;
  float ms = 0;
  cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
  ctx->stats.ms_events += ms;
  cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]);
  ctx->stats.ms_search += ms;
  cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]);
  ctx->stats.ms_sort += ms;
  cudaEventElapsedTime(&ms, ctx->ev[5], ctx->ev[6]);
  ctx->stats.ms_chain += ms;
  ctx->stats.queries += hc.n_queries;
  ctx->stats.hits += hc.n_hits;
  ctx->stats.anchors += n;
  ctx->stats.capped_queries += hc.n_capped;
  ctx->stats.overflow_queries += ctx->search_lean ? hc.n_overflow : hc.n_queries;
  ctx->stats.raw_events += hc.n_events_raw;
  ctx->stats.events += hc.n_events_kept;
  ctx->stats.chunks += Bpres;
  ctx->stats.steps++;
  ctx->stats.linked += hc.n_linked;
  ctx->stats.pending += hc.n_pending;
  if (mode != SORT_GLOBAL) ctx->stats.seg_sort_steps++;
  if (mode == SORT_PART) ctx->stats.part_sort_steps++;
  if (hc.error & 4u) return fail(ctx, SMB_ERR_CAPACITY, "per-read chain scratch overflow");
  if (hc.error & 32u) return fail(ctx, SMB_ERR_CAPACITY, "chain candidate exchange list overflow");
  if (Bpres) {
    double n_est = (double)n;
    if (sharded) n_est = std::max(n_est, ctx->h_ctl.p[2]);
    ctx->est_anchors_per_chunk = 0.5 * ctx->est_anchors_per_chunk + 0.5 * (n_est / Bpres);
    ctx->est_queries_per_chunk = std::max(0.9 * ctx->est_queries_per_chunk, (double)hc.n_queries / Bpres);
  }
  // host mirror of the slots the round asked about
  if (rout && rout->ids && rout->info)
    for (uint32_t i = 0; i < n_ids; ++i) {
      sp.h_events[(*rout->ids)[i]] = (*rout->info)[i].num_events;
      sp.h_nchains[(*rout->ids)[i]] = (*rout->info)[i].n_chains;
    }
  return SMB_OK;
}

// ------------------------------------------------------------------ slot space helpers
static int slots_init(smb_ctx *ctx, SlotSpace &sp, uint32_t n_slots) {
  sp.n_slots = n_slots;
  CK(sp.slots.ensure(std::max(n_slots, 1u)));
  CK(cudaMemsetAsync(sp.slots.p, 0, (size_t)std::max(n_slots, 1u) * sizeof(SlotState), ctx->stream));
  sp.h_events.assign(n_slots, 0);
  sp.h_nchains.assign(n_slots, 0);
  sp.round = 0;
  return SMB_OK;
}

// prepare the out pool of a round: capacity for every participating slot, counters zeroed
static int round_begin(smb_ctx *ctx, SlotSpace &sp, const std::vector<uint32_t> &slots, int step,
                       uint32_t out_pool) {
  uint64_t need_anchor = 0, need_chain = 0;
  const uint32_t max_chains = std::min<uint32_t>(3u * (ctx->index.max_bucket + 1u), 4096u);
  for (uint32_t sl : slots) {
    // a chain has strictly increasing query positions: <= one anchor per seed position
    need_anchor += (uint64_t)(sp.h_events[sl] + kFeatCap) / (uint32_t)std::max(step, 1) + 4ull * max_chains;
    need_chain += max_chains;
  }
  // growing a pool would lose nothing: the out pool holds no live data at round start
  CK(sp.pool_anchor[out_pool].ensure(need_anchor + 64));
  CK(sp.pool_chain[out_pool].ensure(need_chain + 64));
  if (!sp.pool_anchor[1 - out_pool].p) CK(sp.pool_anchor[1 - out_pool].ensure(64));
  if (!sp.pool_chain[1 - out_pool].p) CK(sp.pool_chain[1 - out_pool].ensure(64));
  CK(cudaMemsetAsync(&ctx->d_ctr.p->carry_anchor_used[out_pool], 0, sizeof(unsigned long long), ctx->stream));
  CK(cudaMemsetAsync(&ctx->d_ctr.p->carry_chain_used[out_pool], 0, sizeof(unsigned long long), ctx->stream));
  CK(cudaMemsetAsync(&ctx->d_ctr.p->error, 0, sizeof(unsigned int), ctx->stream));
  return SMB_OK;
}

// run one round over `present` (entries with a chunk) + `absent` slots, splitting into steps;
// what `rout` asks for is read back together with the counters of the round's last step
template <class FillFn>
static int run_round(smb_ctx *ctx, SlotSpace &sp, const std::vector<uint32_t> &present,
                     const std::vector<uint32_t> &absent, StepSource src, const smb_params &prm,
                     FillFn fill /* (StepEntries&, first, count) for present entries */,
                     const RoundOut *rout = nullptr) {
  const uint32_t out_pool = sp.round & 1u;
  std::vector<uint32_t> all(present);
  all.insert(all.end(), absent.begin(), absent.end());
  int rc = round_begin(ctx, sp, all, prm.step_size, out_pool);
  if (rc) return rc;
  // absent slots ride along with the first step (pure copy-forward)
  size_t at = 0;
  bool absent_done = absent.empty();
  const int kbits = bits_for(ctx->index.max_tpos) + bits_for(ctx->index.max_bucket);
  while (at < present.size() || !absent_done) {
    uint32_t max_ev = 0;
    for (size_t i = at; i < present.size(); ++i) max_ev = std::max(max_ev, sp.h_events[present[i]]);
    const int ebits_max = 64 - kbits - bits_for((uint64_t)max_ev + kFeatCap);
    if (ebits_max < 1) return fail(ctx, SMB_ERR_CAPACITY, "sort key does not fit 64 bits");
    uint64_t Bmax = std::min<uint64_t>(ctx->max_batch_chunks, ebits_max >= 31 ? (1ull << 31) : (1ull << ebits_max));
    Bmax = std::min<uint64_t>(Bmax, (1ull << (32 - kQueryBits)) - 1);  // the query payload holds the entry
    uint64_t by_anchors = (uint64_t)(0.6 * (double)ctx->max_batch_anchors / std::max(ctx->est_anchors_per_chunk, 1.0));
    uint32_t count = (uint32_t)std::min<uint64_t>(present.size() - at, std::max<uint64_t>(1, std::min(Bmax, by_anchors)));
    int sort_mode = SORT_PART;
    for (int tries = 0;; ++tries) {
      if (tries > 64) return fail(ctx, SMB_ERR_CAPACITY, "a pipeline step keeps aborting");
      StepEntries en;
      en.B_present = count;
      en.slot.assign(present.begin() + at, present.begin() + at + count);
      fill(en, at, count);
      if (!absent_done) en.slot.insert(en.slot.end(), absent.begin(), absent.end());
      en.B = (uint32_t)en.slot.size();
      const bool last = at + count >= present.size();
      rc = run_step(ctx, sp, en, src, prm, out_pool, &sort_mode, last ? rout : nullptr);
      if (rc == 2) continue;  // aborted on the device, cause dealt with: again
      if (rc == 1) {  // anchor buffer overflow: grow the buffers, or halve the step at the limit
        ctx->est_anchors_per_chunk *= 2.0;
        if ((ctx->ex && ctx->index.sharded) ? ctx->group_at_limit : ctx->last_cap >= ctx->max_batch_anchors) {
          if (count <= 1) return fail(ctx, SMB_ERR_CAPACITY, "one chunk overflows max_batch_anchors");
          count = (count + 1) / 2;
        }
        continue;
      }
      if (rc) return rc;
      break;
    }
    absent_done = true;
    at += count;
  }
  sp.round++;
  return SMB_OK;
}

// Contig-sharded runs: ad/at/aq and the query span of chain 0 are computed by the rank that holds
// chain 0's anchors (SlotState::owned0); everybody else contributes zeros, so a SUM all-reduce
// of the bit patterns hands every rank the owner's values.  flags bit0 (5000-hit cap) is OR-ed.
static int merge_owner_tags(smb_ctx *ctx, std::vector<SlotState> &st, size_t n) {
  if (!ctx->ex || !ctx->index.sharded || n == 0) return SMB_OK;
  std::vector<uint32_t> h(n * 6);
  auto bits = [](float f) { uint32_t u; memcpy(&u, &f, 4); return u; };
  for (size_t r = 0; r < n; ++r) {
    const SlotState &x = st[r];
    const bool own = x.n_chains > 0 && x.owned0;
    h[r * 6 + 0] = own ? bits(x.ad) : 0u;
    h[r * 6 + 1] = own ? bits(x.at) : 0u;
    h[r * 6 + 2] = own ? bits(x.aq) : 0u;
    h[r * 6 + 3] = own ? x.q_first : 0u;
    h[r * 6 + 4] = own ? x.q_last : 0u;
    h[r * 6 + 5] = x.flags & 1u;
  }
  Workspace &w = ctx->ws;
  cudaStream_t s = ctx->stream;
  CK(w.tags.ensure(n * 6));
  CK(cudaMemcpyAsync(w.tags.p, h.data(), n * 6 * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
  int rc = ctx->ex->allreduce(w.tags.p, n * 6, EX_U32, EX_SUM, s, ctx->err);
  if (rc) return rc;
  CK(cudaMemcpyAsync(h.data(), w.tags.p, n * 6 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  ctx->stats.exchanges++;
  auto flt = [](uint32_t u) { float f; memcpy(&f, &u, 4); return f; };
  for (size_t r = 0; r < n; ++r) {
    SlotState &x = st[r];
    x.ad = flt(h[r * 6 + 0]);
    x.at = flt(h[r * 6 + 1]);
    x.aq = flt(h[r * 6 + 2]);
    x.q_first = h[r * 6 + 3];
    x.q_last = h[r * 6 + 4];
    x.flags = (x.flags & ~1u) | (h[r * 6 + 5] ? 1u : 0u);
  }
  return SMB_OK;
}

// ------------------------------------------------------------------ final rows (A.4)
static void make_row(const smb_ctx *ctx, const SlotState &st, uint32_t read_len, uint32_t chunks_used,
                     smb_mapping *m) {
  memset(m, 0, sizeof *m);
  const uint32_t bp_per_sec = 450, sample_rate = 4000, chunk_size = 4000;
  m->read_len = read_len;
  m->chunks = chunks_used;
  m->n_chains = st.n_chains;
  m->num_events = st.num_events;
  m->mapq = 61;  // sigmap.cc:864
  m->flags = st.flags & 1u;
  if (st.n_chains >= 1) {
    m->cm = st.cm;
    m->s1 = st.s1;
    m->s2 = st.s2;
    m->sm = st.sm;
    m->ad = st.ad;
    m->at = st.at;
    m->aq = st.aq;
    if (st.mapped) {
      // sigmap.cc:694-696, :746-766
      volatile float scale_num = (float)chunks_used * chunk_size / st.num_events;
      volatile float scale_den = (float)sample_rate / bp_per_sec;
      const float scale = scale_num / scale_den;
      m->mapped = 1;
      m->q_start = (uint32_t)(scale * st.q_last);
      m->q_end = (uint32_t)(scale * st.q_first);
      m->strand_plus = st.c0_dir;
      m->contig = st.c0_contig;
      const uint32_t clen = st.c0_contig < ctx->contig_len.size() ? ctx->contig_len[st.c0_contig] : 0;
      m->t_start = st.c0_dir ? st.c0_start : (uint32_t)(clen + 1 - st.c0_end);
      m->frag_len = st.c0_end - st.c0_start + 1;
      m->mapq = st.c0_mapq & 63u;
    }
  }
}

// Run-time switches for A/B measurements and for tests that must reach the fallback paths.
// Names are the SMB_<NAME> environment variables (read once by smb_create) without the prefix,
// case-insensitive.  Returns false for an unknown name.
static bool apply_option(smb_ctx *ctx, const char *name_in, const char *value) {
  std::string name(name_in);
  for (char &c : name) c = (char)toupper((unsigned char)c);
  if (name == "SORT") {  // part (default) | entry | global
    ctx->seg_sort = strcmp(value, "global") != 0;
    ctx->part_sort = strcmp(value, "entry") != 0 && ctx->seg_sort;
  } else if (name == "SEARCH") {  // lean (default) | general
    ctx->search_lean = strcmp(value, "general") != 0;
  } else if (name == "FRONT_CAP") {
    ctx->front_cap = (uint32_t)std::max(atoi(value), 0);
  } else if (name == "RUNS_CAP") {
    ctx->runs_cap_min = (uint32_t)std::max(atoi(value), 0);
  } else if (name == "CLOUD_TILE") {  // takes effect at the next device cloud build
    ctx->cloud_tile = (uint32_t)std::min(std::max(atoi(value), 1), 1 << 30);
  } else if (name == "DP_TILES") {
    ctx->dp_pass_max_entries = (uint32_t)std::max(atoi(value), 0);
  } else if (name == "SORT_QUERIES_MIN") {
    ctx->sort_queries_min = (uint32_t)std::max(atoi(value), 0);
  } else if (name == "PIPELINE") {
    ctx->pipeline_mode = strcmp(value, "on") == 0 ? 1 : (strcmp(value, "off") == 0 ? 2 : 0);
  } else if (name == "PREP_ROUNDS") {
    ctx->prep_rounds = std::min(std::max(atoi(value), 0), 200);
  } else if (name == "DP_PASSES") {
    ctx->dp_passes = std::max(atoi(value), 0);
  } else if (name == "UPLOAD_SLICE_MB") {
    ctx->upload_slice_bytes = (size_t)std::max(atoi(value), 1) << 20;
  } else if (name == "EVENTS_OVERLAP") {
    ctx->ev_overlap = strcmp(value, "0") != 0;
  } else if (name == "EVENTS") {  // auto (default) | thread | warp
    ctx->ev_warp_max = !strcmp(value, "thread") ? 0u : (!strcmp(value, "warp") ? 0xFFFFFFFFu : 2048u);
  } else {
    return false;
  }
  return true;
}

// ================================================================== C ABI
extern "C" {

void smb_default_params(smb_params *p) {
  p->search_radius = 0.08f;
  p->step_size = 2;
  p->max_num_chunks = 30;
  p->min_num_anchors = 10;
  p->min_num_anchors_output = 10;
  p->stop_mapping = 1.4f;
  p->stop_mapping_output = 1.2f;
  p->stop_mapping_mean = 5.0f;
  p->stop_mapping_mean_output = 5.0f;
}

int smb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

const char *smb_last_error(const smb_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int smb_create(smb_ctx **out, int device) {
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    g_create_error = "no CUDA device available; sigmap_b200 has no CPU fallback";
    return SMB_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= n) {
    g_create_error = "device index out of range";
    return SMB_ERR_ARG;
  }
  smb_ctx *ctx = new smb_ctx();
  ctx->device = device;
  ctx->front_cap = kFrontCap;
  ctx->dp_passes = kDpFreePasses;
  ctx->prep_rounds = kPrepRounds;
  ctx->dp_pass_max_entries = kDpPassMaxEntries;
  auto bail = [&](const char *what, cudaError_t err) {
    g_create_error = std::string(what) + ": " + cudaGetErrorString(err);
    delete ctx;
    return SMB_ERR_CUDA;
  };
  if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
  if ((e = cudaStreamCreateWithFlags(&ctx->stream.h, cudaStreamNonBlocking)) != cudaSuccess)
    return bail("cudaStreamCreate", e);
  if ((e = ctx->d_ctr.alloc(1)) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = cudaMemset(ctx->d_ctr.p, 0, sizeof(Counters))) != cudaSuccess) return bail("cudaMemset", e);
  if ((e = ctx->h_ctr.alloc(1)) != cudaSuccess || (e = ctx->h_ctl.alloc(4)) != cudaSuccess) return bail("cudaMallocHost", e);
  for (auto &ev : ctx->ev)
    if ((e = cudaEventCreate(&ev.h)) != cudaSuccess) return bail("cudaEventCreate", e);
  for (auto &ev : ctx->timer)
    if ((e = cudaEventCreate(&ev.h)) != cudaSuccess) return bail("cudaEventCreate", e);
  // the per-entry sort keeps a whole part of an entry in shared memory (200 KB of the 227 KB)
  if ((e = cudaFuncSetAttribute(k_seg_sort<kSortCapBig, 1024, 8192>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)sort_smem_bytes(kSortCapBig, 8192))) != cudaSuccess)
    return bail("cudaFuncSetAttribute(k_seg_sort)", e);
  // the general search kernel keeps one stack per index level in shared memory: from 7 levels on
  // (> 16.7 M points, i.e. references beyond ~8 Mbp) a CTA needs more than the default 48 KB; the
  // lean one holds the top levels and its warps' frontiers in up to 208 KB
  {
    const int need = (int)(kSearchWarps * search_smem_per_warp(kMaxLevels));
    if ((e = cudaFuncSetAttribute(k_radius_search<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, need)) != cudaSuccess ||
        (e = cudaFuncSetAttribute(k_radius_search<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, need)) != cudaSuccess)
      return bail("cudaFuncSetAttribute(k_radius_search)", e);
    const int lean = (int)kLeanSmemLimit;  // the staging buffers take what the staged top levels leave
    static_assert(kTopSmemMax + kLeanWarps * kLeanWarpSmem + 1024 <= 232448, "lean search kernel: 227 KB of shared memory per SM");
    if ((e = cudaFuncSetAttribute(k_search_lean<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lean)) != cudaSuccess ||
        (e = cudaFuncSetAttribute(k_search_lean<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lean)) != cudaSuccess)
      return bail("cudaFuncSetAttribute(k_search_lean)", e);
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
    ctx->n_sm = (unsigned)n_sm;
  }
  if ((e = cudaFuncSetAttribute(k_part_sort<kPartSortCap, 512, 4096>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)part_sort_smem_bytes(kPartSortCap, 4096))) != cudaSuccess)
    return bail("cudaFuncSetAttribute(k_part_sort)", e);
  for (const char *name : {"SORT", "SEARCH", "FRONT_CAP", "RUNS_CAP", "DP_PASSES", "DP_TILES", "SORT_QUERIES_MIN",
                           "PREP_ROUNDS", "PIPELINE", "EVENTS_OVERLAP", "EVENTS", "UPLOAD_SLICE_MB", "CLOUD_TILE"})
    if (const char *env = getenv((std::string("SMB_") + name).c_str())) apply_option(ctx, name, env);
  {
    int per_sm = 0, n_sm = 148;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_chain_dp, kDpThreads, 0) != cudaSuccess || per_sm < 1)
      per_sm = 8;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
    ctx->dp_grid = (unsigned)(per_sm * n_sm);
  }
  if ((e = cudaFuncSetAttribute(k_ev_chunk_warp<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)kEvWarpSmem)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(k_ev_chunk_warp<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)kEvWarpSmem)) != cudaSuccess)
    return bail("cudaFuncSetAttribute(k_ev_chunk_warp)", e);
  if ((e = cudaStreamCreateWithFlags(&ctx->stream_ev.h, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&ctx->stream_cp.h, cudaStreamNonBlocking)) != cudaSuccess)
    return bail("cudaStreamCreate", e);
  for (int c = 0; c < 2; ++c)
    if ((e = cudaEventCreate(&ctx->ev_blk_t0[c].h)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev_blk_t1[c].h)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->ev_cp[c].h)) != cudaSuccess)
      return bail("cudaEventCreate", e);
  if ((e = cudaEventCreateWithFlags(&ctx->ev_input.h, cudaEventDisableTiming)) != cudaSuccess)
    return bail("cudaEventCreate", e);
  *out = ctx;
  return SMB_OK;
}

void smb_destroy(smb_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  cudaStreamSynchronize(ctx->stream_ev);
  cudaStreamSynchronize(ctx->stream_cp);
  smb_stream_close(ctx);
  delete ctx;
}

void smb_stats_reset(smb_ctx *ctx) { memset(&ctx->stats, 0, sizeof ctx->stats); }

int smb_stats_get(smb_ctx *ctx, smb_stats *out) {
  ctx->stats.ms_total = ctx->stats.ms_events + ctx->stats.ms_search + ctx->stats.ms_sort +
                        ctx->stats.ms_chain + ctx->stats.ms_filter;
  *out = ctx->stats;
  return SMB_OK;
}

int smb_timer_start(smb_ctx *ctx) {
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventRecord(ctx->timer[0], ctx->stream));
  return SMB_OK;
}

int smb_timer_stop(smb_ctx *ctx, double *ms) {
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventRecord(ctx->timer[1], ctx->stream));
  CK(cudaEventSynchronize(ctx->timer[1]));
  float f = 0;
  CK(cudaEventElapsedTime(&f, ctx->timer[0], ctx->timer[1]));
  *ms = f;
  return SMB_OK;
}

int smb_set_limits(smb_ctx *ctx, uint32_t max_batch_chunks, uint64_t max_batch_anchors) {
  if (max_batch_chunks) ctx->max_batch_chunks = max_batch_chunks;
  if (max_batch_anchors) {
    if (max_batch_anchors >= (1ull << 30)) return fail(ctx, SMB_ERR_ARG, "max_batch_anchors must be < 2^30");
    ctx->max_batch_anchors = max_batch_anchors;
  }
  return SMB_OK;
}

int smb_set_option(smb_ctx *ctx, const char *name, const char *value) {
  if (!name || !value) return fail(ctx, SMB_ERR_ARG, "smb_set_option: null name or value");
  if (!apply_option(ctx, name, value)) return fail(ctx, SMB_ERR_ARG, std::string("smb_set_option: unknown option ") + name);
  return SMB_OK;
}

// ---------------------------------------------------------- contig-sharded runs
int smbh_assign_contigs(const uint32_t *lengths, uint32_t n_contigs, uint32_t world, uint32_t *owner) {
  if (world == 0) return SMB_ERR_ARG;
  // longest-processing-time bin packing: contigs by decreasing length onto the lightest rank
  std::vector<uint32_t> order(n_contigs);
  for (uint32_t c = 0; c < n_contigs; ++c) order[c] = c;
  std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return lengths[x] > lengths[y]; });
  std::vector<uint64_t> load(world, 0);
  for (uint32_t c : order) {
    uint32_t best = 0;
    for (uint32_t r = 1; r < world; ++r)
      if (load[r] < load[best]) best = r;
    owner[c] = best;
    load[best] += lengths[c];
  }
  return SMB_OK;
}

int smb_shard_local_group(smb_ctx *const *ctxs, uint32_t n) {
  if (n == 0) return SMB_ERR_ARG;
  auto g = std::make_shared<LocalGroup>();
  g->world = (int)n;
  g->send.assign(n, nullptr);
  g->device.resize(n);
  for (uint32_t r = 0; r < n; ++r) g->device[r] = ctxs[r]->device;
  for (uint32_t r = 0; r < n; ++r) {
    // peers on other GPUs: direct loads over NVLink when the driver allows it
    cudaSetDevice(ctxs[r]->device);
    for (uint32_t q = 0; q < n; ++q) {
      int can = 0;
      if (ctxs[q]->device != ctxs[r]->device &&
          cudaDeviceCanAccessPeer(&can, ctxs[r]->device, ctxs[q]->device) == cudaSuccess && can)
        if (cudaDeviceEnablePeerAccess(ctxs[q]->device, 0) != cudaSuccess) cudaGetLastError();
    }
    auto ex = std::make_unique<LocalExchange>();
    ex->rank = (int)r;
    ex->world = (int)n;
    ex->g = g;
    ex->device = ctxs[r]->device;
    ctxs[r]->ex = std::move(ex);
    ctxs[r]->local_group = g;
  }
  return SMB_OK;
}

int smb_shard_nccl_unique_id(char *id128) {
  NcclApi &api = NcclApi::get();
  if (!api.load()) {
    g_create_error = api.error;
    return SMB_ERR_STATE;
  }
  NcclApi::unique_id id;
  const int rc = api.GetUniqueId(&id);
  if (rc != 0) {
    g_create_error = std::string("ncclGetUniqueId: ") + api.GetErrorString(rc);
    return SMB_ERR_CUDA;
  }
  memcpy(id128, id.internal, 128);
  return SMB_OK;
}

int smb_shard_nccl_init(smb_ctx *ctx, int rank, int world, const char *id128) {
  CK(cudaSetDevice(ctx->device));
  if (world < 1 || rank < 0 || rank >= world) return fail(ctx, SMB_ERR_ARG, "bad rank / world");
  NcclApi &api = NcclApi::get();
  if (!api.load()) return fail(ctx, SMB_ERR_STATE, api.error);
  NcclApi::unique_id id;
  memcpy(id.internal, id128, 128);
  auto ex = std::make_unique<NcclExchange>();
  ex->rank = rank;
  ex->world = world;
  const int rc = api.CommInitRank(&ex->comm, world, id, rank);
  if (rc != 0) return fail(ctx, SMB_ERR_CUDA, std::string("ncclCommInitRank: ") + api.GetErrorString(rc));
  ctx->ex = std::move(ex);
  return SMB_OK;
}

int smb_shard_rank(const smb_ctx *ctx) { return ctx->ex ? ctx->ex->rank : 0; }
int smb_shard_world(const smb_ctx *ctx) { return ctx->ex ? ctx->ex->world : 1; }

// ------------------------------------------------------------ whole hot path
}  // extern "C"

// device buffers and the per-read tables of a read set (everything but the samples and where they
// lie), on stream s.  pack_off (n_reads + 1): the reads laid end to end, which lays out `kept`.
static int reads_prepare(smb_ctx *ctx, const uint64_t *pack_off, const float *dig, const float *range,
                         const float *offset, size_t n_reads, cudaStream_t s) {
  ctx->n_reads = n_reads;
  if (n_reads == 0) return SMB_OK;
  if (n_reads > 0xFFFFFFF0ull) return fail(ctx, SMB_ERR_ARG, "too many reads");
  const uint64_t total = pack_off[n_reads];
  ctx->h_kept_off.resize(n_reads);
  ctx->h_offset.assign(offset, offset + n_reads);
  ctx->h_scale.resize(n_reads);
  for (size_t r = 0; r < n_reads; ++r) {
    // 64-sample (128-byte) aligned, non-overlapping regions: the events kernel loads int4
    ctx->h_kept_off[r] = ((pack_off[r] + 63) & ~63ull) + 64ull * r;
    ctx->h_scale[r] = range[r] / dig[r];  // float / float as signal_batch.cc:195
  }
  const uint64_t kept_total = ((total + 63) & ~63ull) + 64ull * n_reads + 64;
  CK(ctx->kept.ensure(kept_total));
  CK(ctx->d_kept_off.ensure(n_reads));
  CK(ctx->d_dig.ensure(n_reads));
  CK(ctx->d_range.ensure(n_reads));
  CK(ctx->d_offset.ensure(n_reads));
  CK(ctx->d_kept_len.ensure(n_reads));
  CK(ctx->h_kept_pinned.ensure(n_reads));
  CK(cudaMemcpyAsync(ctx->d_kept_off.p, ctx->h_kept_off.data(), n_reads * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(ctx->d_dig.p, dig, n_reads * sizeof(float), cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(ctx->d_range.p, range, n_reads * sizeof(float), cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(ctx->d_offset.p, offset, n_reads * sizeof(float), cudaMemcpyHostToDevice, s));
  ctx->stats.h2d_bytes += n_reads * 20;
  return SMB_OK;
}

// reads_prepare for samples that the call copies from the host into `raw`: read_off goes up as
// K1's offset table
static int reads_prepare_host(smb_ctx *ctx, const uint64_t *read_off, const float *dig, const float *range,
                              const float *offset, size_t n_reads, cudaStream_t s) {
  ctx->device_input = false;
  const int rc = reads_prepare(ctx, read_off, dig, range, offset, n_reads, s);
  if (rc || n_reads == 0) return rc;
  CK(ctx->raw.ensure(read_off[n_reads] + 8));
  CK(ctx->d_read_off.ensure(n_reads + 1));
  CK(cudaMemcpyAsync(ctx->d_read_off.p, read_off, (n_reads + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
  ctx->stats.h2d_bytes += n_reads * 8 + 8;
  return SMB_OK;
}

extern "C" {

int smb_reads_upload(smb_ctx *ctx, const int16_t *raw, const uint64_t *read_off, const float *dig,
                     const float *range, const float *offset, size_t n_reads) {
  CK(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  int rc = reads_prepare_host(ctx, read_off, dig, range, offset, n_reads, s);
  if (rc || n_reads == 0) return rc;
  const uint64_t total = read_off[n_reads];
  CK(cudaMemcpyAsync(ctx->raw.p, raw, total * sizeof(int16_t), cudaMemcpyHostToDevice, s));
  ctx->stats.h2d_bytes += total * 2;
  CK(cudaStreamSynchronize(s));
  return SMB_OK;
}

}  // extern "C"

// K1's input: read r is raw[beg[r] .. end[r]).  host != nullptr (smb_map_reads): the call first
// copies the samples from host, packed as host_off says, into raw, slice by slice.
struct ReadSource {
  const int16_t *raw;
  const uint64_t *beg, *end;
  const int16_t *host = nullptr;
  const uint64_t *host_off = nullptr;
};

// the samples of smb_reads_upload / smb_map_reads, packed in `raw` as read_off says
static ReadSource uploaded_source(const smb_ctx *ctx) {
  return {ctx->raw.p, ctx->d_read_off.p, ctx->d_read_off.p + 1};
}

// K1 over reads [r0, r1) on stream s: (30,200) pA filter + compaction, kept lengths to the
// pinned host mirror (no wait here)
static int filter_slice(smb_ctx *ctx, const ReadSource &src, size_t r0, size_t r1, cudaStream_t s) {
  if (r1 <= r0) return SMB_OK;
  k_filter_compact<<<(unsigned)(r1 - r0), kFilterThreads, 0, s>>>(src.raw, src.beg + r0, src.end + r0, ctx->d_dig.p + r0,
                                                                ctx->d_range.p + r0, ctx->d_offset.p + r0,
                                                                ctx->d_kept_off.p + r0, ctx->kept.p,
                                                                ctx->d_kept_len.p + r0, (uint32_t)(r1 - r0));
  LAUNCH_CHECK();
  CK(cudaMemcpyAsync(ctx->h_kept_pinned.p + r0, ctx->d_kept_len.p + r0, (r1 - r0) * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  ctx->stats.d2h_bytes += (r1 - r0) * 4;
  return SMB_OK;
}

// The read set as the copy stream delivers it to the mapping loop.  Slice k = reads
// [first_read[k], first_read[k+1]); done[k] fires once the slice's samples are on the device, have
// been filtered, and its kept lengths are in the pinned host mirror.
struct UploadPlan {
  std::vector<size_t> first_read;
  std::vector<cudaEvent_t> done;
  size_t admitted = 0;  // slices handed to the mapping loop so far
  bool pending() const { return admitted < done.size(); }
};

// from construction to destruction no cudaFree (it waits for the whole device, i.e. for the queued
// slices): a buffer that grows parks its old allocation
struct DeferFrees {
  DeferFrees() { FreeLater::on = true; }
  ~DeferFrees() {
    FreeLater::on = false;
    FreeLater::drain();
  }
};

static int slice_event(smb_ctx *ctx, size_t k, cudaEvent_t *out) {
  while (k >= ctx->slice_events.size()) {
    Event e;
    if (cudaEventCreateWithFlags(&e.h, cudaEventDisableTiming) != cudaSuccess)
      return fail(ctx, SMB_ERR_CUDA, "cudaEventCreate (upload slice)");
    ctx->slice_events.push_back(std::move(e));
  }
  *out = ctx->slice_events[k];
  return SMB_OK;
}

// Enqueues the read set on the copy stream in slices of consecutive reads, each: [its samples
// copied from src.host] -> K1 over its reads -> kept lengths to the host -> its done event, with
// ev_cp[0] / ev_cp[1] around all of them.  A slice takes one read, then more while they fit in
// slice_samples (host input: as read_off packs them; otherwise in the kept layout);
// slice_samples = 0: one slice of every read.
static int plan_slices(smb_ctx *ctx, const ReadSource &src, uint64_t slice_samples, UploadPlan &plan) {
  const size_t R = ctx->n_reads;
  cudaStream_t cs = ctx->stream_cp;
  CK(cudaEventRecord(ctx->ev_cp[0], cs));
  for (size_t r0 = 0, r1; r0 < R; r0 = r1) {
    r1 = slice_samples ? r0 + 1 : R;
    if (src.host)
      while (r1 < R && src.host_off[r1 + 1] - src.host_off[r0] <= slice_samples) ++r1;
    else
      while (r1 < R && ctx->h_kept_off[r1] - ctx->h_kept_off[r0] <= slice_samples) ++r1;
    cudaEvent_t done;
    int rc = slice_event(ctx, plan.done.size(), &done);
    if (rc) return rc;
    if (src.host) {
      const uint64_t a = src.host_off[r0], b = src.host_off[r1];
      const cudaError_t ce =
          cudaMemcpyAsync(ctx->raw.p + a, src.host + a, (b - a) * sizeof(int16_t), cudaMemcpyHostToDevice, cs);
      if (ce != cudaSuccess) return fail(ctx, SMB_ERR_CUDA, std::string("upload slice: ") + cudaGetErrorString(ce));
      ctx->stats.h2d_bytes += (b - a) * 2;
    }
    rc = filter_slice(ctx, src, r0, r1, cs);
    if (rc) return rc;
    CK(cudaEventRecord(done, cs));
    plan.first_read.push_back(r0);
    plan.done.push_back(done);
  }
  plan.first_read.push_back(R);
  CK(cudaEventRecord(ctx->ev_cp[1], cs));
  return SMB_OK;
}

// K1 time of a read set filtered on the copy stream (not for host input, whose slices also copy)
static int add_filter_time(smb_ctx *ctx) {
  CK(cudaEventSynchronize(ctx->ev_cp[1]));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, ctx->ev_cp[0], ctx->ev_cp[1]));
  ctx->stats.ms_filter += ms;
  return SMB_OK;
}

// Event detection does not depend on the mapping state, only on the raw signal, and its kernels
// are one-thread-per-chunk sequential scans that want as many chunks per launch as possible.  So
// events run in LOOKAHEAD BLOCKS: the next `depth` chunks of every read active at tick r0 in one
// launch, cached as feature rows (two feature caches, so that the next block can be computed on
// the event stream while the ticks of the current one are being mapped; a block is handed over
// with a host wait on its event).
struct EvBlock {
  uint32_t r0 = 0, r1 = 0;            // ticks covered
  bool ready = false;                 // launched, not yet consumed
  std::vector<uint32_t> row_base;     // per read: first row of the read in the block's cache
  std::vector<uint64_t> cs;           // host chunk table (kept alive until the block is consumed)
  std::vector<float> co, csc;
};
constexpr uint32_t kEvRowCap = 96u << 10;

// The read scheduler of a mapping call, which advances in TICKS: tick t maps the next chunk of
// every active read.  Reads join ("are admitted") at a tick boundary, slice by slice as the copy
// stream delivers them, so read r is at chunk t - t_admit[r]; which reads share a tick changes the
// composition of the batches, never a row.  The two tick policies, run_blocks and run_waves, work
// on this state.
struct Sched {
  smb_ctx *ctx;
  SlotSpace &sp;
  const smb_params &prm;
  const size_t R;
  UploadPlan plan;
  std::vector<uint32_t> n_chunks, chunks_used, t_admit;
  uint32_t round = 0;                          // the tick
  std::vector<RoundInfo> info;                 // of the reads of the last tick
  uint64_t first_active = 0, after_first = 0;  // reads that had a first chunk / went past it
  EvBlock blk[2];
  int cur = 0;  // the block the ticks read

  Sched(smb_ctx *c, SlotSpace &s, const smb_params &p)
      : ctx(c), sp(s), prm(p), R(c->n_reads), n_chunks(R, 0), chunks_used(R, 1), t_admit(R, 0) {}

  uint32_t chunk_limit(uint32_t r) const { return std::min<uint32_t>(n_chunks[r], (uint32_t)prm.max_num_chunks); }

  // Takes the plan's next slice if it has arrived (wait: once it has).  Its kept lengths go to
  // h_kept_len and n_chunks, and its reads that have a whole chunk to map to `into`.  *took =
  // false: no slice is left, or the next one has not arrived.
  int take_slice(bool wait, std::vector<uint32_t> &into, bool *took) {
    *took = false;
    if (!plan.pending()) return SMB_OK;
    const size_t k = plan.admitted;
    const cudaError_t q = cudaEventQuery(plan.done[k]);
    if (q == cudaErrorNotReady) {
      if (!wait) return SMB_OK;
      ctx->stats.sync_points++;
      CK(cudaEventSynchronize(plan.done[k]));
    } else if (q != cudaSuccess) {
      return fail(ctx, SMB_ERR_CUDA, std::string("upload slice: ") + cudaGetErrorString(q));
    }
    for (size_t r = plan.first_read[k]; r < plan.first_read[k + 1]; ++r) {
      ctx->h_kept_len[r] = ctx->h_kept_pinned.p[r];
      n_chunks[r] = ctx->h_kept_len[r] / kChunk;  // tail dropped, sigmap.cc:643
      if (n_chunks[r] > 0 && prm.max_num_chunks > 0) into.push_back((uint32_t)r);
    }
    plan.admitted++;
    *took = true;
    return SMB_OK;
  }

  // the end of a tick that mapped `act` (info[i] is act[i]'s): chunks used, the survival counts,
  // and the reads that go on to another chunk appended to `next`
  void end_tick(const std::vector<uint32_t> &act, std::vector<uint32_t> &next) {
    ctx->stats.samples += (uint64_t)act.size() * kChunk;
    for (size_t i = 0; i < act.size(); ++i) {
      const uint32_t r = act[i];
      const uint32_t done = round + 1 - t_admit[r];
      chunks_used[r] = done;
      const bool more = !info[i].stop && done < n_chunks[r] && done < (uint32_t)prm.max_num_chunks;
      if (done == 1) {
        ++first_active;
        if (more) ++after_first;
      }
      if (more) next.push_back(r);
    }
    ++round;
  }

  // enqueue the events of ticks [r0, r0 + depth) of `who` on the event stream, into cache `c`
  int launch_block(int c, uint32_t r0, uint32_t depth, const std::vector<uint32_t> &who) {
    EvBlock &b = blk[c];
    Workspace &w = ctx->ws;
    cudaStream_t s = ctx->stream_ev;
    b.r0 = r0;
    b.r1 = r0 + depth;
    b.row_base.assign(R, 0);
    b.cs.clear();
    b.co.clear();
    b.csc.clear();
    for (uint32_t r : who) {
      b.row_base[r] = (uint32_t)b.cs.size();
      const uint32_t c0 = r0 - t_admit[r];  // the read's chunk at tick r0
      const uint32_t lim = std::min(chunk_limit(r), c0 + depth);
      for (uint32_t ch = c0; ch < lim; ++ch) {
        b.cs.push_back(ctx->h_kept_off[r] + (uint64_t)kChunk * ch);
        b.co.push_back(ctx->h_offset[r]);
        b.csc.push_back(ctx->h_scale[r]);
      }
    }
    const uint32_t rows = (uint32_t)b.cs.size();
    CK(cudaEventRecord(ctx->ev_blk_t0[c], s));
    if (rows) {
      CK(w.blk_chunk_start.ensure(rows));
      CK(w.blk_chunk_offset.ensure(rows));
      CK(w.blk_chunk_scale.ensure(rows));
      CK(w.feat_cache[c].ensure((size_t)rows * kFeatCap));
      CK(w.nf_cache[c].ensure(rows));
      CK(w.nraw_cache[c].ensure(rows));
      CK(cudaMemcpyAsync(w.blk_chunk_start.p, b.cs.data(), rows * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
      CK(cudaMemcpyAsync(w.blk_chunk_offset.p, b.co.data(), rows * sizeof(float), cudaMemcpyHostToDevice, s));
      CK(cudaMemcpyAsync(w.blk_chunk_scale.p, b.csc.data(), rows * sizeof(float), cudaMemcpyHostToDevice, s));
      ctx->stats.h2d_bytes += rows * 16ull;
      const ChunkTable ct{w.blk_chunk_start.p, w.blk_chunk_offset.p, w.blk_chunk_scale.p};
      int rc = run_events(ctx, SRC_RAW_KEPT, ctx->kept.p, rows, nullptr, w.feat_cache[c].p, w.nf_cache[c].p,
                          w.nraw_cache[c].p, s, &ct);
      if (rc) return rc;
    }
    CK(cudaEventRecord(ctx->ev_blk_t1[c], s));
    b.ready = true;
    return SMB_OK;
  }

  // wait for block `c` and make it the one the ticks read
  int consume_block(int c) {
    ctx->stats.sync_points++;
    CK(cudaEventSynchronize(ctx->ev_blk_t1[c]));
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev_blk_t0[c], ctx->ev_blk_t1[c]);
    ctx->stats.ms_events += ms;
    blk[c].ready = false;
    cur = c;
    ctx->ws.cache_cur = c;
    return SMB_OK;
  }
};

// Ticks in lookahead event blocks.  A block is several ticks deep only while most reads survive
// from tick to tick (full-read mapping), one tick deep when the stop rules retire most reads after
// their first chunk or while reads are still being admitted.  The kernels are latency-bound and
// leave the SMs almost idle, so the NEXT block is computed while the current one is being mapped.
static int run_blocks(Sched &S) {
  smb_ctx *ctx = S.ctx;
  std::vector<uint32_t> active;
  const std::vector<uint32_t> none;
  bool have_next = false;  // blk[1 - cur] holds a launched block for round == blk[cur].r1
  size_t prev_active = 0;
  int rc;
  bool took;
  // contig shards must run identical ticks on every rank: no timing-dependent admission
  if (ctx->ex && ctx->index.sharded)
    while (S.plan.pending()) {
      rc = S.take_slice(true, active, &took);
      if (rc) return rc;
    }
  while (!active.empty() || S.plan.pending()) {
    const uint32_t round = S.round;
    if (round >= S.blk[S.cur].r1) {
      // a block boundary: the only place reads are admitted (every row of a block then belongs
      // to a read that was there when the block was launched).  Wait for a slice only when no
      // read is active.
      const size_t n0 = active.size();
      bool wait = active.empty();
      do {
        rc = S.take_slice(wait, active, &took);
        if (rc) return rc;
        wait = false;  // one is enough to go on; take whatever else is ready
      } while (took);
      for (size_t i = n0; i < active.size(); ++i) S.t_admit[active[i]] = round;
      if (active.empty()) continue;  // that slice held no read with a whole chunk
      // (a prefetched block is only ever launched once every slice has been admitted, so it
      // covers every read that is active now)
      if (have_next && S.blk[1 - S.cur].r0 == round) {
        rc = S.consume_block(1 - S.cur);
        if (rc) return rc;
      } else {
        uint32_t depth = 1;
        if (round > 0 && !S.plan.pending() && active.size() * 2 > prev_active)
          depth = (uint32_t)std::min<size_t>(8, std::max<size_t>(1, kEvRowCap / active.size()));
        const int c = round == 0 ? 0 : 1 - S.cur;
        rc = S.launch_block(c, round, depth, active);
        if (rc) return rc;
        rc = S.consume_block(c);
        if (rc) return rc;
      }
      have_next = false;
    }
    // the block after this one, while this one is being mapped: worth it only while most reads
    // go on from tick to tick (known from the previous tick; for tick 0 from the last call) and
    // nobody is waiting to be admitted
    if (ctx->ev_overlap && !have_next && !S.plan.pending()) {
      const bool surviving = round > 0 ? active.size() * 2 > prev_active : ctx->ev_survival_hint > 0.5;
      if (surviving) {
        const uint32_t r0n = S.blk[S.cur].r1;
        std::vector<uint32_t> who;
        who.reserve(active.size());
        for (uint32_t r : active)
          if (S.chunk_limit(r) > r0n - S.t_admit[r]) who.push_back(r);
        if (!who.empty()) {
          const uint32_t depth = (uint32_t)std::min<size_t>(8, std::max<size_t>(1, kEvRowCap / who.size()));
          rc = S.launch_block(1 - S.cur, r0n, depth, who);
          if (rc) return rc;
          have_next = true;
        }
      }
    }
    prev_active = active.size();
    const std::vector<uint32_t> &row_base = S.blk[S.cur].row_base;
    const uint32_t ev_r0 = S.blk[S.cur].r0;
    auto fill = [&](StepEntries &en, size_t first, uint32_t count) {
      en.feat_row.resize(count);
      for (uint32_t i = 0; i < count; ++i) en.feat_row[i] = row_base[active[first + i]] + (round - ev_r0);
    };
    RoundOut rout;
    rout.ids = &active;
    rout.info = &S.info;
    rc = run_round(ctx, S.sp, active, none, SRC_CACHED, S.prm, fill, &rout);
    if (rc) return rc;
    std::vector<uint32_t> next;
    next.reserve(active.size());
    S.end_tick(active, next);
    active.swap(next);
  }
  return SMB_OK;
}

// Wave-pipelined ticks.  Every tick maps the reads of ONE event block (one tick deep); while it is
// being mapped, the block of the next tick is computed on the event stream for the reads that are
// known by then: the survivors of the PREVIOUS tick (they wait one tick, carried forward as absent
// slots) and the reads whose slices have arrived since -- at most one step's worth.  So neither K1
// nor event detection is ever waited for after the first wave, however the reads arrive.  A read's
// chunk at tick T is T - t_admit[r]; t_admit is (re)set whenever the read is put into a block, which
// is all that "waiting a tick" takes.
static int run_waves(Sched &S) {
  smb_ctx *ctx = S.ctx;
  std::vector<uint32_t> done_chunks(S.R, 0), members[2], waiting, absent;
  auto want_reads = [&]() -> size_t {
    const uint64_t by_anchors = (uint64_t)(0.6 * (double)ctx->max_batch_anchors / std::max(ctx->est_anchors_per_chunk, 1.0));
    return (size_t)std::max<uint64_t>(1, std::min<uint64_t>(by_anchors, ctx->max_batch_chunks));
  };
  // reads of the slices that have arrived, in order, until `cap` have joined; wait: block until at
  // least `min_new` have joined or no slice is left
  auto join = [&](std::vector<uint32_t> &into, size_t min_new, size_t cap, bool wait) -> int {
    const size_t n0 = into.size();
    for (bool took = true; took && into.size() - n0 < cap;) {
      const int rc = S.take_slice(wait && into.size() - n0 < min_new, into, &took);
      if (rc) return rc;
    }
    return SMB_OK;
  };
  auto launch_for = [&](int c, uint32_t tick) -> int {
    for (uint32_t r : members[c]) S.t_admit[r] = tick - done_chunks[r];
    return S.launch_block(c, tick, 1, members[c]);
  };
  int c = 0, rc;
  bool have_blk = false;  // blk[c] has been launched for tick `round` with members[c]
  for (;;) {
    if (!have_blk) {
      // nothing was prefetched for this tick: whoever is waiting, plus new reads (a batch, or
      // what is left of the input)
      members[c].swap(waiting);
      waiting.clear();
      const size_t want = want_reads();
      if (members[c].size() < want && S.plan.pending()) {
        const size_t room = want - members[c].size();
        rc = join(members[c], (room + 1) / 2, room, true);
        if (rc) return rc;
      }
      if (members[c].empty()) {
        if (!S.plan.pending()) break;
        continue;  // slices without a single whole chunk
      }
      rc = launch_for(c, S.round);
      if (rc) return rc;
    }
    rc = S.consume_block(c);
    if (rc) return rc;
    have_blk = false;
    const std::vector<uint32_t> &act = members[c];
    // the next tick's block while this one is mapped
    absent.clear();
    for (uint32_t r : waiting)
      if (S.sp.h_nchains[r] > 0) absent.push_back(r);
    if (ctx->ev_overlap) {
      std::vector<uint32_t> &nx = members[1 - c];
      nx.swap(waiting);
      waiting.clear();
      const size_t want = want_reads();
      if (nx.size() < want && S.plan.pending()) {
        rc = join(nx, 0, want - nx.size(), false);
        if (rc) return rc;
      }
      if (!nx.empty()) {
        rc = launch_for(1 - c, S.round + 1);
        if (rc) return rc;
        have_blk = true;
      }
    }
    const std::vector<uint32_t> &row_base = S.blk[c].row_base;
    auto fill = [&](StepEntries &en, size_t first, uint32_t count) {
      en.feat_row.resize(count);
      for (uint32_t i = 0; i < count; ++i) en.feat_row[i] = row_base[act[first + i]];
    };
    RoundOut rout;
    rout.ids = &act;
    rout.info = &S.info;
    rc = run_round(ctx, S.sp, act, absent, SRC_CACHED, S.prm, fill, &rout);
    if (rc) return rc;
    S.end_tick(act, waiting);
    for (uint32_t r : waiting) done_chunks[r] = S.chunks_used[r];
    if (have_blk) c = 1 - c;
  }
  return SMB_OK;
}

// what every mapping entry point checks before it does any work
static int map_check(smb_ctx *ctx, const smb_params *prm) {
  if (!ctx->has_index) return fail(ctx, SMB_ERR_STATE, "no index loaded");
  if (prm->step_size < 1) return fail(ctx, SMB_ERR_ARG, "step_size must be >= 1");
  return SMB_OK;
}

// Maps the read set (ctx->n_reads reads, their samples where `src` says): every mapping entry
// point ends here, after map_check.
static int map_read_set(smb_ctx *ctx, const smb_params *prm_in, smb_mapping *out, const ReadSource &src) {
  CK(cudaSetDevice(ctx->device));
  const smb_params prm = *prm_in;
  const size_t R = ctx->n_reads;
  // Wave-pipelined ticks when the stop rules retire most reads after their first chunk (known from
  // the previous call; a fresh context starts this way): K1 and the events of the next wave run
  // while the current one is being mapped (option pipeline=on: also with resident samples, which
  // then join in waves of filter-only slices).  Contig shards must run identical ticks on every
  // rank: no timing-dependent admission there.
  // auto: only when the samples arrive from the host during the call.  With resident samples the
  // GPU is busy mapping from the first tick on and the overlap only adds contention and steps
  // (measured on config 3: 437 ms pipelined against 403 ms; with host buffers on two GPUs e2e
  // 1.65 against 1.58 G samples/s).
  const bool sharded_index = ctx->ex && ctx->index.sharded;
  const bool pipeline = !sharded_index && R > 0 && prm.max_num_chunks > 0 &&
                        (ctx->pipeline_mode == 1 ||
                         (ctx->pipeline_mode == 0 && src.host && ctx->ev_survival_hint <= 0.5));
  Sched S(ctx, ctx->map_slots, prm);
  int rc = slots_init(ctx, S.sp, (uint32_t)R);
  if (rc) return rc;
  // Slices still queued when the mapping starts (host input, or wave-pipelined): frees wait for
  // the end of the mapping.  The one slice of any other call is waited for before the first tick.
  const bool sliced = src.host || pipeline;
  std::optional<DeferFrees> defer;
  if (sliced) defer.emplace();
  rc = plan_slices(ctx, src, sliced ? ctx->upload_slice_bytes / sizeof(int16_t) : 0, S.plan);
  if (rc) return rc;
  ctx->h_kept_len.resize(R);
  rc = pipeline ? run_waves(S) : run_blocks(S);
  if (rc) return rc;
  // a block launched for ticks that never came (every read stopped) must not outlive the call
  if (S.blk[0].ready || S.blk[1].ready) CK(cudaStreamSynchronize(ctx->stream_ev));
  if (S.first_active) ctx->ev_survival_hint = (double)S.after_first / (double)S.first_active;
  if (!src.host && R) {
    rc = add_filter_time(ctx);
    if (rc) return rc;
  }
  // final rows
  std::vector<SlotState> st(std::max<size_t>(R, 1));
  if (R) {
    CK(cudaMemcpyAsync(st.data(), S.sp.slots.p, R * sizeof(SlotState), cudaMemcpyDeviceToHost, ctx->stream));
    rc = host_sync(ctx);
    if (rc) return rc;
    ctx->stats.d2h_bytes += R * sizeof(SlotState);
    rc = merge_owner_tags(ctx, st, R);
    if (rc) return rc;
  }
  for (size_t r = 0; r < R; ++r) make_row(ctx, st[r], ctx->h_kept_len[r], S.chunks_used[r], &out[r]);
  return SMB_OK;
}

// The end of every mapping call: nothing of it stays queued on the copy stream.  Nothing of a
// failed call stays queued on the other two streams either (the caller of smb_map_reads_device may
// free raw once the call returns), and a failed member must not leave its in-process peers waiting
// at a rendezvous.
static int map_done(smb_ctx *ctx, int rc) {
  cudaStreamSynchronize(ctx->stream_cp);
  if (rc) {
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->stream_ev);
    if (ctx->local_group) ctx->local_group->abort_all();
  }
  return rc;
}

// raw must be device (or managed) memory of this context's device
static int check_device_input(smb_ctx *ctx, const void *raw) {
  cudaPointerAttributes a{};
  const cudaError_t e = cudaPointerGetAttributes(&a, raw);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(ctx, SMB_ERR_ARG, std::string("raw: cudaPointerGetAttributes: ") + cudaGetErrorString(e));
  }
  if (a.type == cudaMemoryTypeUnregistered)
    return fail(ctx, SMB_ERR_ARG, "raw is pageable host memory, not device memory (host samples go through smb_map_reads)");
  if (a.type == cudaMemoryTypeHost)
    return fail(ctx, SMB_ERR_ARG, "raw is pinned host memory, not device memory (host samples go through smb_map_reads)");
  if (a.device != ctx->device)
    return fail(ctx, SMB_ERR_ARG, "raw is memory of device " + std::to_string(a.device) + ", this context runs on device " +
                                      std::to_string(ctx->device));
  return SMB_OK;
}

static int map_device_impl(smb_ctx *ctx, const int16_t *raw, const uint64_t *read_start, const uint32_t *read_len,
                           const float *dig, const float *range, const float *offset, size_t n_reads,
                           const smb_params *params, smb_mapping *out, cudaStream_t caller) {
  CK(cudaSetDevice(ctx->device));
  int rc = map_check(ctx, params);
  if (rc) return rc;
  // pack: the reads laid end to end (the kept layout); span: K1's start table, then its end table
  std::vector<uint64_t> pack(n_reads + 1, 0), span(2 * n_reads);
  for (size_t r = 0; r < n_reads; ++r) {
    pack[r + 1] = pack[r] + read_len[r];
    span[r] = read_start[r];
    span[n_reads + r] = read_start[r] + read_len[r];
  }
  if (pack[n_reads]) {  // raw is not read when every read is empty
    rc = check_device_input(ctx, raw);
    if (rc) return rc;
  }
  // the context's streams do not synchronise with the legacy default stream (NULL): it is waited
  // for like any other
  cudaStream_t s = ctx->stream;
  CK(cudaEventRecord(ctx->ev_input, caller));
  CK(cudaStreamWaitEvent(s, ctx->ev_input, 0));
  ctx->device_input = true;
  rc = reads_prepare(ctx, pack.data(), dig, range, offset, n_reads, s);
  if (rc) return rc;
  if (n_reads) {
    CK(ctx->d_read_off.ensure(2 * n_reads));
    CK(cudaMemcpyAsync(ctx->d_read_off.p, span.data(), 2 * n_reads * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += n_reads * 16;
    // K1 runs on the copy stream, after the tables
    CK(cudaEventRecord(ctx->ev_input, s));
    CK(cudaStreamWaitEvent(ctx->stream_cp, ctx->ev_input, 0));
  }
  return map_read_set(ctx, params, out, {raw, ctx->d_read_off.p, ctx->d_read_off.p + n_reads});
}

extern "C" {

int smb_map_uploaded(smb_ctx *ctx, const smb_params *prm_in, smb_mapping *out) {
  if (ctx->device_input)
    return fail(ctx, SMB_ERR_STATE, "no uploaded reads: the last read set was mapped from device memory "
                                    "(smb_map_reads_device); upload one with smb_reads_upload or smb_map_reads");
  const int rc = map_check(ctx, prm_in);
  if (rc) return rc;
  return map_done(ctx, map_read_set(ctx, prm_in, out, uploaded_source(ctx)));
}

int smb_map_reads(smb_ctx *ctx, const int16_t *raw, const uint64_t *read_off, const float *dig,
                  const float *range, const float *offset, size_t n_reads, const smb_params *params,
                  smb_mapping *out) {
  CK(cudaSetDevice(ctx->device));
  // the small per-read tables first, then the samples in slices of ~64 MB on the copy stream:
  // copy -> K1 filter of the slice's reads -> kept lengths to the host -> event.  The mapping loop
  // admits a slice's reads once its event has fired, so the rest of the upload hides behind the
  // mapping of the reads that are already there (raw should be pinned host memory for that).
  int rc = map_check(ctx, params);
  if (rc) return rc;
  rc = reads_prepare_host(ctx, read_off, dig, range, offset, n_reads, ctx->stream_cp);
  if (!rc) {
    ReadSource src = uploaded_source(ctx);
    src.host = raw;
    src.host_off = read_off;
    rc = map_read_set(ctx, params, out, src);
  }
  return map_done(ctx, rc);
}

int smb_map_reads_device(smb_ctx *ctx, const int16_t *raw, const uint64_t *read_start, const uint32_t *read_len,
                         const float *digitisation, const float *range, const float *offset, size_t n_reads,
                         const smb_params *params, smb_mapping *out, void *stream) {
  return map_done(ctx, map_device_impl(ctx, raw, read_start, read_len, digitisation, range, offset, n_reads,
                                       params, out, (cudaStream_t)stream));
}

// ------------------------------------------------------------- stage hooks
int smb_stage_raw_to_pa(smb_ctx *ctx, const int16_t *raw, size_t n, float dig, float offset, float range,
                        float *out, size_t *n_out) {
  CK(cudaSetDevice(ctx->device));
  uint64_t off[2] = {0, n};
  int rc = smb_reads_upload(ctx, raw, off, &dig, &range, &offset, 1);
  if (rc) return rc;
  UploadPlan plan;  // K1 in one slice
  rc = plan_slices(ctx, uploaded_source(ctx), 0, plan);
  if (rc) return rc;
  ctx->stats.sync_points++;
  CK(cudaEventSynchronize(plan.done[0]));
  rc = add_filter_time(ctx);
  if (rc) return rc;
  const uint32_t kept = ctx->h_kept_pinned.p[0];
  *n_out = kept;
  if (!kept) return SMB_OK;
  DevBuf<float> d;
  CK(d.ensure(kept));
  k_raw_to_pa<<<(kept + 255) / 256, 256, 0, ctx->stream>>>(ctx->kept.p + ctx->h_kept_off[0], kept, offset,
                                                          ctx->h_scale[0], d.p);
  LAUNCH_CHECK();
  CK(cudaMemcpyAsync(out, d.p, kept * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return SMB_OK;
}

static int stage_events_common(smb_ctx *ctx, const float *pa, size_t n_chunks, uint32_t *d_peaks) {
  Workspace &w = ctx->ws;
  cudaStream_t s = ctx->stream;
  const uint32_t B = (uint32_t)n_chunks;
  DevBuf<float> d_pa;
  CK(d_pa.ensure((size_t)B * kChunk));
  CK(cudaMemcpyAsync(d_pa.p, pa, (size_t)B * kChunk * sizeof(float), cudaMemcpyHostToDevice, s));
  std::vector<uint64_t> start(B);
  for (uint32_t b = 0; b < B; ++b) start[b] = (uint64_t)b * kChunk;
  CK(w.chunk_start.ensure(B));
  CK(w.n_features.ensure(B));
  CK(w.n_raw_events.ensure(B));
  CK(w.features.ensure((size_t)B * kFeatCap));
  CK(cudaMemcpyAsync(w.chunk_start.p, start.data(), B * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
  int rc = run_events(ctx, SRC_PA_FLOAT, d_pa.p, B, d_peaks);
  if (rc) return rc;
  CK(cudaStreamSynchronize(s));
  return SMB_OK;
}

int smb_stage_events(smb_ctx *ctx, const float *pa, size_t n_chunks, float *features, uint32_t *n_features) {
  CK(cudaSetDevice(ctx->device));
  if (n_chunks == 0) return SMB_OK;
  int rc = stage_events_common(ctx, pa, n_chunks, nullptr);
  if (rc) return rc;
  CK(cudaMemcpy(features, ctx->ws.features.p, n_chunks * kFeatCap * sizeof(float), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(n_features, ctx->ws.n_features.p, n_chunks * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  return SMB_OK;
}

int smb_stage_detect(smb_ctx *ctx, const float *pa, float *tstat1, float *tstat2, uint32_t *peaks,
                     uint32_t *n_peaks, float *means, uint32_t *n_events) {
  CK(cudaSetDevice(ctx->device));
  DevBuf<uint32_t> d_peaks;
  CK(d_peaks.ensure(kFeatCap));
  int rc = stage_events_common(ctx, pa, 1, d_peaks.p);
  if (rc) return rc;
  const uint32_t Bp = 32;
  uint32_t ne = 0;
  CK(cudaMemcpy(&ne, ctx->ws.n_raw_events.p, sizeof(uint32_t), cudaMemcpyDeviceToHost));
  if (n_events) *n_events = ne;
  if (n_peaks) *n_peaks = ne;  // #events == #peaks (the last peak only closes the count)
  if (tstat1) CK(cudaMemcpy2D(tstat1, sizeof(float), ctx->ws.t1.p, Bp * sizeof(float), sizeof(float), kChunk + 1, cudaMemcpyDeviceToHost));
  if (tstat2) CK(cudaMemcpy2D(tstat2, sizeof(float), ctx->ws.t2.p, Bp * sizeof(float), sizeof(float), kChunk + 1, cudaMemcpyDeviceToHost));
  if (peaks && ne) CK(cudaMemcpy(peaks, d_peaks.p, ne * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  if (means && ne) CK(cudaMemcpy(means, ctx->ws.means.p, ne * sizeof(float), cudaMemcpyDeviceToHost));
  return SMB_OK;
}

int smb_stage_radius(smb_ctx *ctx, const float *queries, size_t nq, float radius, uint64_t *hit_off,
                     uint64_t *hit_idx, float *hit_d2, uint64_t cap) {
  CK(cudaSetDevice(ctx->device));
  if (!ctx->has_index) return fail(ctx, SMB_ERR_STATE, "no index loaded");
  if (nq > 0xFFFFFFF0ull) return fail(ctx, SMB_ERR_ARG, "too many queries");
  cudaStream_t s = ctx->stream;
  hit_off[0] = 0;
  if (nq == 0) return SMB_OK;
  DevBuf<float> d_q, d_a, d_b;
  DevBuf<uint64_t> k_a, k_b;
  DevBuf<unsigned long long> cnt;
  DevBuf<unsigned char> tmp;
  const uint64_t dcap = std::max<uint64_t>(cap, 1);
  CK(d_q.ensure(nq * kDim));
  CK(k_a.ensure(dcap));
  CK(k_b.ensure(dcap));
  CK(d_a.ensure(dcap));
  CK(d_b.ensure(dcap));
  CK(cnt.ensure(nq));
  CK(cudaMemcpyAsync(d_q.p, queries, nq * kDim * sizeof(float), cudaMemcpyHostToDevice, s));
  k_reset_step<<<1, 1, 0, s>>>(ctx->d_ctr.p);
  LAUNCH_CHECK();
  SearchArgs sa{};
  sa.features = d_q.p;
  sa.n_queries = (uint32_t)nq;
  sa.radius = radius;
  sa.out_key = k_a.p;
  sa.out_dist = d_a.p;
  sa.cap = dcap;
  sa.ctr = ctx->d_ctr.p;
  {
    int rc = launch_search<true>(ctx, sa, (uint32_t)nq, s);
    if (rc) return rc;
  }
  CK(cudaMemcpyAsync(ctx->h_ctr.p, ctx->d_ctr.p, sizeof(Counters), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  const unsigned long long n = ctx->h_ctr.p->n_anchors;
  if (n > cap) return fail(ctx, SMB_ERR_CAPACITY, "smb_stage_radius: more hits than cap");
  CK(cudaMemsetAsync(cnt.p, 0, nq * sizeof(unsigned long long), s));
  const uint64_t *keys = k_a.p;
  const float *dd = d_a.p;
  if (n > 1) {
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, k_a.p, k_b.p, d_a.p, d_b.p, (uint64_t)n, 0, 64, s);
    CK(tmp.ensure(tb));
    CK(cub::DeviceRadixSort::SortPairs(tmp.p, tb, k_a.p, k_b.p, d_a.p, d_b.p, (uint64_t)n, 0, 64, s));
    keys = k_b.p;
    dd = d_b.p;
  }
  if (n > 0) {
    k_count_by_query<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(keys, n, cnt.p);
    LAUNCH_CHECK();
  }
  std::vector<unsigned long long> h_cnt(nq);
  std::vector<uint64_t> h_keys(n);
  CK(cudaMemcpyAsync(h_cnt.data(), cnt.p, nq * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
  if (n) {
    CK(cudaMemcpyAsync(h_keys.data(), keys, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(hit_d2, dd, n * sizeof(float), cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  for (size_t q = 0; q < nq; ++q) hit_off[q + 1] = hit_off[q] + h_cnt[q];
  for (unsigned long long i = 0; i < n; ++i) hit_idx[i] = h_keys[i] & 0xFFFFFFFFull;
  return SMB_OK;
}

// ------------------------------------------------------------- batch of read slots
int smb_batch_create(smb_ctx *ctx, uint32_t n_slots, smb_batch **batch) {
  CK(cudaSetDevice(ctx->device));
  smb_batch *b = new smb_batch{ctx, {}};
  int rc = slots_init(ctx, b->sp, n_slots);
  if (rc) {
    delete b;
    return rc;
  }
  *batch = b;
  return SMB_OK;
}

void smb_batch_destroy(smb_batch *b) {
  if (!b) return;
  cudaSetDevice(b->ctx->device);
  cudaStreamSynchronize(b->ctx->stream);
  delete b;
}

int smb_batch_reset(smb_batch *b) { return slots_init(b->ctx, b->sp, b->sp.n_slots); }

int smb_batch_generate_chains(smb_batch *b, const uint32_t *slots, uint32_t n, const float *features,
                              const uint32_t *feat_off, const smb_params *prm) {
  smb_ctx *ctx = b->ctx;
  CK(cudaSetDevice(ctx->device));
  if (prm->step_size < 1) return fail(ctx, SMB_ERR_ARG, "step_size must be >= 1");
  std::vector<uint32_t> present(slots, slots + n), absent;
  std::vector<uint8_t> seen(b->sp.n_slots, 0);
  for (uint32_t i = 0; i < n; ++i) {
    if (slots[i] >= b->sp.n_slots || seen[slots[i]]) return fail(ctx, SMB_ERR_ARG, "bad or repeated slot");
    seen[slots[i]] = 1;
  }
  for (uint32_t sl = 0; sl < b->sp.n_slots; ++sl)
    if (!seen[sl] && b->sp.h_nchains[sl] > 0) absent.push_back(sl);
  DevBuf<float> d_feat;
  DevBuf<uint32_t> d_off;
  const uint32_t total = feat_off[n];
  CK(d_feat.ensure(std::max(total, 1u)));
  CK(d_off.ensure(n + 1));
  CK(cudaMemcpyAsync(d_feat.p, features, total * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  std::vector<uint32_t> rel(n + 1);
  auto fill = [&](StepEntries &en, size_t first, uint32_t count) {
    // offsets of this step's slice, rebased so the device sees [first, first+count]
    for (uint32_t i = 0; i <= count; ++i) rel[i] = feat_off[first + i];
    cudaMemcpyAsync(d_off.p, rel.data(), (count + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream);
    en.d_features = d_feat.p;
    en.d_feat_off = d_off.p;
  };
  std::vector<RoundInfo> info;
  std::vector<uint32_t> all(present);
  all.insert(all.end(), absent.begin(), absent.end());
  RoundOut rout;
  rout.ids = &all;
  rout.info = &info;
  int rc = run_round(ctx, b->sp, present, absent, SRC_FEATURES, *prm, fill, &rout);
  cudaStreamSynchronize(ctx->stream);
  return rc;
}

static int slot_state(smb_batch *b, uint32_t slot, SlotState *st) {
  smb_ctx *ctx = b->ctx;
  if (slot >= b->sp.n_slots) return fail(ctx, SMB_ERR_ARG, "slot out of range");
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpy(st, b->sp.slots.p + slot, sizeof(SlotState), cudaMemcpyDeviceToHost));
  return SMB_OK;
}

int smb_batch_chain_count(smb_batch *b, uint32_t slot, uint32_t *n_chains) {
  SlotState st;
  int rc = slot_state(b, slot, &st);
  if (rc) return rc;
  *n_chains = st.n_chains;
  return SMB_OK;
}

int smb_batch_get_chains(smb_batch *b, uint32_t slot, smb_chain *out, uint32_t cap) {
  smb_ctx *ctx = b->ctx;
  SlotState st;
  int rc = slot_state(b, slot, &st);
  if (rc) return rc;
  const uint32_t n = std::min(cap, st.n_chains);
  std::vector<ChainRec> recs(std::max(n, 1u));
  if (n) CK(cudaMemcpy(recs.data(), b->sp.pool_chain[st.pool].p + st.chain_off, n * sizeof(ChainRec), cudaMemcpyDeviceToHost));
  for (uint32_t i = 0; i < n; ++i)
    out[i] = smb_chain{recs[i].score, recs[i].contig, recs[i].start, recs[i].end, recs[i].n_anchors,
                       recs[i].mapq, recs[i].dir};
  return SMB_OK;
}

int smb_batch_get_anchors(smb_batch *b, uint32_t slot, uint32_t chain, smb_anchor *out, uint32_t cap) {
  smb_ctx *ctx = b->ctx;
  SlotState st;
  int rc = slot_state(b, slot, &st);
  if (rc) return rc;
  if (chain >= st.n_chains) return fail(ctx, SMB_ERR_ARG, "chain out of range");
  ChainRec rec;
  CK(cudaMemcpy(&rec, b->sp.pool_chain[st.pool].p + st.chain_off + chain, sizeof(ChainRec), cudaMemcpyDeviceToHost));
  if (rec.anchor_off == 0xFFFFFFFFu) return fail(ctx, SMB_ERR_STATE, "the chain's anchors live on the rank that owns its contig");
  const uint32_t n = std::min(cap, rec.n_anchors);
  std::vector<CarryAnchor> an(std::max(n, 1u));
  if (n) CK(cudaMemcpy(an.data(), b->sp.pool_anchor[st.pool].p + st.carry_off + rec.anchor_off, n * sizeof(CarryAnchor), cudaMemcpyDeviceToHost));
  for (uint32_t i = 0; i < n; ++i) out[i] = smb_anchor{an[i].target, an[i].query, an[i].dist};
  return SMB_OK;
}

// ---------------------------------------------------------------- streaming
// Channels keep, on the host, the filtered remainder that does not yet fill a chunk (H9:
// chunk boundaries are defined on the filtered stream); completed chunks of all channels are
// mapped as one round.
int smb_stream_open(smb_ctx *ctx, uint32_t n_channels, const smb_params *params) {
  CK(cudaSetDevice(ctx->device));
  if (!ctx->has_index) return fail(ctx, SMB_ERR_STATE, "no index loaded");
  if (ctx->stream_slots) smb_stream_close(ctx);
  ctx->stream_slots = std::make_unique<SlotSpace>();
  int rc = slots_init(ctx, *ctx->stream_slots, n_channels);
  if (rc) return rc;
  ctx->stream_params = *params;
  ctx->stream_pending.assign(n_channels, {});
  ctx->stream_offset.assign(n_channels, 0.f);
  ctx->stream_scale.assign(n_channels, 1.f);
  ctx->stream_chunks.assign(n_channels, 0);
  ctx->stream_kept.assign(n_channels, 0);
  ctx->stream_lo.assign(n_channels, 0);
  ctx->stream_hi.assign(n_channels, -1);
  ctx->stream_generic.assign(n_channels, 1);
  return SMB_OK;
}

int smb_stream_close(smb_ctx *ctx) {
  if (ctx->stream_slots) {
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->stream_slots.reset();
  }
  ctx->h_stream_stage.release();
  ctx->d_stream_stage.release();
  return SMB_OK;
}

// the K1 filter of one raw value on the host: same fp32 expression as raw_to_pa()
static inline bool host_keep(int raw, float off, float scale) {
  volatile float sum = (float)raw + off;  // volatile: two separately rounded fp32 operations
  volatile float pa = sum * scale;
  return pa > 30.0f && pa < 200.0f;
}

// Raw values kept on a channel.  For finite offset and finite positive scale the conversion
// fl(fl(raw + offset) * scale) is non-decreasing in raw, so "pA > 30" holds from some raw value
// upwards and "pA < 200" up to some raw value: two binary searches over the int16 range.
static void stream_keep_interval(float off, float scale, int32_t &lo, int32_t &hi, uint8_t &generic) {
  generic = !(scale > 0.0f) || !std::isfinite(scale) || !std::isfinite(off);
  lo = 0;
  hi = -1;
  if (generic) return;
  auto above30 = [&](int raw) {
    volatile float sum = (float)raw + off;
    volatile float pa = sum * scale;
    return pa > 30.0f;
  };
  auto below200 = [&](int raw) {
    volatile float sum = (float)raw + off;
    volatile float pa = sum * scale;
    return pa < 200.0f;
  };
  int a = -32768, b = 32768;  // first raw in [a, b) with above30, b if none
  while (a < b) {
    const int m = a + (b - a) / 2;
    if (above30(m)) b = m; else a = m + 1;
  }
  lo = a;
  a = -32769, b = 32767;      // last raw in (a, b] with below200, a if none
  while (a < b) {
    const int m = b - (b - a) / 2;
    if (below200(m)) a = m; else b = m - 1;
  }
  hi = a;
}

int smb_stream_begin_read(smb_ctx *ctx, uint32_t ch, float dig, float range, float offset) {
  if (!ctx->stream_slots || ch >= ctx->stream_slots->n_slots) return fail(ctx, SMB_ERR_ARG, "bad channel");
  CK(cudaSetDevice(ctx->device));
  SlotSpace &sp = *ctx->stream_slots;
  CK(cudaMemsetAsync(sp.slots.p + ch, 0, sizeof(SlotState), ctx->stream));
  sp.h_events[ch] = 0;
  sp.h_nchains[ch] = 0;
  ctx->stream_pending[ch].clear();
  ctx->stream_offset[ch] = offset;
  ctx->stream_scale[ch] = range / dig;
  ctx->stream_chunks[ch] = 0;
  ctx->stream_kept[ch] = 0;
  stream_keep_interval(offset, ctx->stream_scale[ch], ctx->stream_lo[ch], ctx->stream_hi[ch],
                       ctx->stream_generic[ch]);
  return SMB_OK;
}

int smb_stream_round(smb_ctx *ctx, const uint32_t *channels, uint32_t n, const int16_t *samples,
                     const uint32_t *sample_off, uint8_t *decisions, smb_mapping *maps) {
  if (!ctx->stream_slots) return fail(ctx, SMB_ERR_STATE, "stream not open");
  CK(cudaSetDevice(ctx->device));
  SlotSpace &sp = *ctx->stream_slots;
  const smb_params &prm = ctx->stream_params;
  // host-side range filter of the incoming samples (same decisions as K1) and chunk cutting;
  // completed chunks go straight into the pinned staging buffer
  if ((size_t)n * kChunk > ctx->h_stream_stage.cap) CK(ctx->h_stream_stage.alloc((size_t)std::max(n, sp.n_slots) * kChunk));
  const auto t_stage0 = std::chrono::steady_clock::now();
  std::vector<uint32_t> present;
  present.reserve(n);
  {
    // a channel named twice would put two chunks of one read into the same round
    std::vector<uint8_t> named(sp.n_slots, 0);
    for (uint32_t i = 0; i < n; ++i) {
      if (channels[i] >= sp.n_slots) return fail(ctx, SMB_ERR_ARG, "bad channel");
      if (named[channels[i]]) return fail(ctx, SMB_ERR_ARG, "channel named twice in one round");
      named[channels[i]] = 1;
    }
  }
  // Channels are independent (each named once), so filtering and chunk cutting run on all host
  // cores; channel i's chunk goes to staging slot i and the slots of the channels that completed
  // a chunk are closed up afterwards (nothing moves when every channel did: the usual round).
  std::vector<uint8_t> ready(n, 0);
#pragma omp parallel for schedule(static) if (n >= 64)
  for (int64_t ii = 0; ii < (int64_t)n; ++ii) {
    const uint32_t i = (uint32_t)ii;
    const uint32_t ch = channels[i];
    std::vector<int16_t> &pend = ctx->stream_pending[ch];
    const int16_t *in = samples + sample_off[i];
    const size_t cnt = sample_off[i + 1] - sample_off[i];
    int16_t *slot = ctx->h_stream_stage.p + (size_t)i * kChunk;
    const bool wants = ctx->stream_chunks[ch] < (uint32_t)prm.max_num_chunks;
    bool clean = false;
    if (!ctx->stream_generic[ch]) {
      const int lo = ctx->stream_lo[ch], hi = ctx->stream_hi[ch];
      int outside = 0;
      for (size_t k = 0; k < cnt; ++k) outside |= (in[k] < lo) | (in[k] > hi);
      clean = !outside;
    }
    if (clean && wants && pend.empty() && cnt >= (size_t)kChunk) {
      // nothing filtered, nothing left over: the chunk goes straight from the caller's buffer
      memcpy(slot, in, kChunk * sizeof(int16_t));
      pend.assign(in + kChunk, in + cnt);
      ready[i] = 1;
      continue;
    }
    if (ctx->stream_generic[ch]) {
      const float off = ctx->stream_offset[ch], scale = ctx->stream_scale[ch];
      for (size_t k = 0; k < cnt; ++k)
        if (host_keep(in[k], off, scale)) pend.push_back(in[k]);
    } else if (clean) {
      pend.insert(pend.end(), in, in + cnt);
    } else {
      const int lo = ctx->stream_lo[ch], hi = ctx->stream_hi[ch];
      const size_t old = pend.size();
      pend.resize(old + cnt);
      int16_t *w = pend.data() + old;
      for (size_t k = 0; k < cnt; ++k) {
        *w = in[k];
        w += (in[k] >= lo) & (in[k] <= hi);
      }
      pend.resize((size_t)(w - pend.data()));
    }
    if (pend.size() >= (size_t)kChunk && wants) {
      memcpy(slot, pend.data(), kChunk * sizeof(int16_t));
      pend.erase(pend.begin(), pend.begin() + kChunk);
      ready[i] = 1;
    } else if (!wants) {
      // the read has used up its chunks (sigmap.cc:647): nothing more will be mapped, so the
      // samples are only counted (read length of the row), not buffered
      ctx->stream_kept[ch] += (uint32_t)pend.size();
      pend.clear();
    }
  }
  for (uint32_t i = 0; i < n; ++i) {
    if (!ready[i]) continue;
    if (present.size() != i)
      memmove(ctx->h_stream_stage.p + present.size() * kChunk, ctx->h_stream_stage.p + (size_t)i * kChunk, kChunk * sizeof(int16_t));
    present.push_back(channels[i]);
  }
  ctx->stats.ms_stream_stage +=
      std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_stage0).count();
  // all other channels with live chains are carried forward
  std::vector<uint8_t> seen(sp.n_slots, 0);
  for (uint32_t ch : present) seen[ch] = 1;
  std::vector<uint32_t> absent;
  for (uint32_t ch = 0; ch < sp.n_slots; ++ch)
    if (!seen[ch] && sp.h_nchains[ch] > 0) absent.push_back(ch);
  // decisions + provisional rows for the channels named in this call come back with the round
  std::vector<RoundInfo> info;
  std::vector<uint32_t> everyone(present);
  everyone.insert(everyone.end(), absent.begin(), absent.end());
  std::vector<SlotState> st;
  if (!present.empty() || !absent.empty()) {
    const size_t n_stage = present.size() * kChunk;
    CK(ctx->d_stream_stage.ensure(std::max<size_t>(n_stage, 8)));
    if (n_stage)
      CK(cudaMemcpyAsync(ctx->d_stream_stage.p, ctx->h_stream_stage.p, n_stage * sizeof(int16_t),
                         cudaMemcpyHostToDevice, ctx->stream));
    ctx->stats.h2d_bytes += n_stage * 2;
    auto fill = [&](StepEntries &en, size_t first, uint32_t count) {
      en.samples = ctx->d_stream_stage.p;
      en.chunk_start.resize(count);
      en.offset.resize(count);
      en.scale.resize(count);
      for (uint32_t i = 0; i < count; ++i) {
        const uint32_t ch = present[first + i];
        en.chunk_start[i] = (uint64_t)(first + i) * kChunk;
        en.offset[i] = ctx->stream_offset[ch];
        en.scale[i] = ctx->stream_scale[ch];
      }
    };
    RoundOut rout;
    rout.ids = &everyone;
    rout.info = &info;
    rout.states = &st;
    int rc = run_round(ctx, sp, present, absent, SRC_RAW_KEPT, prm, fill, &rout);
    if (rc) return rc;
    ctx->stats.samples += (uint64_t)present.size() * kChunk;
    for (uint32_t ch : present) {
      ctx->stream_chunks[ch]++;
      ctx->stream_kept[ch] += kChunk;
    }
  } else {
    // nothing to map this round: provisional rows from the slots as they are
    st.resize(std::max<size_t>(sp.n_slots, 1));
    if (sp.n_slots) CK(cudaMemcpy(st.data(), sp.slots.p, sp.n_slots * sizeof(SlotState), cudaMemcpyDeviceToHost));
    ctx->stats.d2h_bytes += sp.n_slots * sizeof(SlotState);
  }
  int rc = merge_owner_tags(ctx, st, sp.n_slots);
  if (rc) return rc;
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t ch = channels[i];
    const bool mapped_chunk = seen[ch] != 0;
    if (decisions) decisions[i] = (mapped_chunk && st[ch].stop) ? 1 : 0;
    if (maps) {
      const uint32_t used = std::max(ctx->stream_chunks[ch], 1u);
      make_row(ctx, st[ch], ctx->stream_kept[ch] + (uint32_t)ctx->stream_pending[ch].size(), used, &maps[i]);
    }
  }
  return SMB_OK;
}

}  // extern "C"
