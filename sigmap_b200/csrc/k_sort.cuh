// k_sort.cuh -- K5: per-entry (per read chunk) anchor sort in shared memory.
//
// The reference sorts every (strand, contig) bucket of one chunk with std::sort on
// (target, query, distance) (spatial_index.cc:411-417, key spatial_index.h:22-25).  A global
// radix sort of the whole batch moves every 12-byte anchor through HBM six times.  Here the
// search kernel already knows which chunk ("entry") a hit belongs to and records where it wrote
// each run of hits (RunRec), so the sort never has to look at the entry bits: ONE CTA per
// entry gathers the entry's runs into its 227 KB of shared memory, sorts them there and writes
// every anchor back exactly once, in (bucket, target, query) order.
//
//   pass 0   (only if the entry does not fit at once) coarse histogram of the linear coordinate
//            g = bucket_base[bucket] + target over <= 256 bins -> contiguous parts of <= kSortCap
//   per part gather (filter by g range) into shared memory + fine histogram (8192 bins)
//            -> exclusive scan -> counting-sort scatter of 16-bit slots -> each bin (1.1 anchors
//            on average) ordered by full key: insertion sort by one thread, or a warp-wide rank
//            sort for the few dense bins (the true locus, carried chains)
//            -> coalesced write-back at a position reserved with one atomic per entry.
//
// Output segments of different entries land in arrival order; inside an entry the order is the
// reference's.  Nothing downstream depends on the order of entries (k_chain_prep finds segment
// bounds from key changes).  (target, query) pairs are unique inside a bucket, so the order is
// total and the result is bit-identical to the radix-sort path.
#ifndef SB_K_SORT_CUH
#define SB_K_SORT_CUH

#include "sb_device.cuh"

namespace sb {

constexpr int kRunsCap = 512;        // run records a k_part_sort CTA holds in shared memory at a time (one tile of a
                                     // list); the lists themselves hold runs_cap records, sized per step by the host
// k_seg_sort runs as <10240, 1024, 8192> (template parameters CAP = anchors of one part held in
// shared memory, THREADS, BINS = fine bins per part): one 200 KB CTA per SM, the fewest passes
// over an entry's runs
constexpr int kSortCapBig = 10240;
// k_part_sort runs as <5120, 512, 4096>: two 105 KB CTAs per SM
constexpr int kPartSortCap = 5120;   // anchors of one (entry, part) held by a k_part_sort CTA
constexpr int kSmallBin = 24;        // bins up to this size: insertion sort by one thread
constexpr int kBigBinCap = 512;      // dense bins queued for the warp-wide rank sort

struct SegSortArgs {
  const uint64_t *key_in;
  const float *dist_in;
  uint64_t *key_out;
  float *dist_out;
  const RunRec *runs;           // [B * n_parts][runs_cap]
  const uint32_t *run_count;    // [B * n_parts]
  uint32_t runs_cap;            // run records per list
  uint32_t n_parts;             // run lists per entry (k_part_sort's partition; 1 = one list)
  uint32_t B;
  KeyLayout kl;
  const uint64_t *bucket_base;  // [n_buckets + 1] linear coordinate of target 0 of each bucket
  int gshift;                   // coarse bin = g >> gshift, < kCoarseBins
  uint32_t n_coarse;
  Counters *ctr;                // sort_cursor (output position), error bit 4 (dense coarse bin)
};

constexpr size_t sort_smem_bytes(int cap, int bins) {
  return (size_t)cap * (8 + 4 + 2 + 2) + (size_t)bins * 4 + (size_t)kCoarseBins * 4 +
         (size_t)(kCoarseBins + 2) * 4 + (size_t)kBigBinCap * 4 + 64 * 4;
}

template <int kSortCap, int kSortThreads, int kSortBins>
__global__ void __launch_bounds__(kSortThreads, kSortThreads == 1024 ? 1 : 2) k_seg_sort(const SegSortArgs a) {
  static_assert(kSortBins % kSortThreads == 0, "bins per thread");
  extern __shared__ __align__(16) unsigned char s_raw[];
  uint64_t *s_key = reinterpret_cast<uint64_t *>(s_raw);
  float *s_dist = reinterpret_cast<float *>(s_key + kSortCap);
  uint32_t *s_bins = reinterpret_cast<uint32_t *>(s_dist + kSortCap);
  uint32_t *s_coarse = s_bins + kSortBins;
  uint32_t *s_part = s_coarse + kCoarseBins;      // [kCoarseBins + 2] part boundaries (coarse bins)
  uint32_t *s_big = s_part + kCoarseBins + 2;     // [kBigBinCap]
  uint32_t *s_misc = s_big + kBigBinCap;          // [64]: 0..31 warp sums, 32 n, 33 nbig, 34 np, 35 total, 36/37 base
  uint16_t *s_order = reinterpret_cast<uint16_t *>(s_misc + 64);
  uint16_t *s_order2 = s_order + kSortCap;

  const uint32_t entry = blockIdx.x;
  if (a.ctr->abort) return;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const unsigned full = 0xffffffffu;
  const unsigned lt = (1u << lane) - 1u;
  // the entry's runs: the lists of its n_parts parts, addressed as one virtual list of
  // n_parts * runs_cap slots (slot v = list v / runs_cap, run v % runs_cap; unused slots skipped)
  const uint32_t rcap = a.runs_cap;
  const RunRec *runs = a.runs + (size_t)entry * a.n_parts * rcap;
  const uint32_t *rcount = a.run_count + (size_t)entry * a.n_parts;
  const uint32_t nr = a.n_parts == 1 ? min(rcount[0], rcap) : a.n_parts * rcap;
  auto run_at = [&](uint32_t v) -> RunRec {
    const uint32_t used = min(rcount[v / rcap], rcap);
    return (v % rcap) < used ? runs[v] : RunRec{0u, 0u};
  };
  const KeyLayout kl = a.kl;

  // ---- total anchors of the entry
  uint32_t mine = 0;
  for (uint32_t r = tid; r < nr; r += kSortThreads) mine += run_at(r).count;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) mine += __shfl_xor_sync(full, mine, d);
  if (tid < kCoarseBins) s_coarse[tid] = 0;
  if (tid < 32) s_misc[tid] = 0;
  __syncthreads();
  if (lane == 0) s_misc[wid] = mine;
  __syncthreads();
  if (wid == 0) {
    uint32_t v = s_misc[lane];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(full, v, d);
    if (lane == 0) s_misc[35] = v;
  }
  __syncthreads();
  const uint32_t total = s_misc[35];
  if (total == 0) return;

  auto coord = [&](uint64_t k) -> uint64_t { return __ldg(a.bucket_base + kl.bucket(k)) + kl.target(k); };

  // ---- pass 0: coarse histogram and the split into parts that fit shared memory
  if (total > (uint32_t)kSortCap) {
    for (uint32_t r = wid; r < nr; r += kSortThreads / 32) {
      const RunRec run = run_at(r);
      for (uint32_t i0 = 0; i0 < run.count; i0 += 4 * 32) {  // a run is <= 128 hits: one trip
        uint64_t kq[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t i = i0 + u * 32 + lane;
          kq[u] = i < run.count ? a.key_in[run.start + i] : ~0ull;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (kq[u] != ~0ull) atomicAdd(&s_coarse[(uint32_t)(coord(kq[u]) >> a.gshift)], 1u);
      }
    }
    __syncthreads();
    if (tid == 0) {
      uint32_t np = 0, acc = 0;
      bool dense = false;
      s_part[0] = 0;
      for (uint32_t b = 0; b < a.n_coarse; ++b) {
        const uint32_t cb = s_coarse[b];
        if (cb > (uint32_t)kSortCap) dense = true;
        if (acc + cb > (uint32_t)kSortCap) {
          s_part[++np] = b;
          acc = 0;
        }
        acc += cb;
      }
      s_part[++np] = a.n_coarse;
      s_misc[34] = dense ? 0u : np;
      if (dense) {  // the host redoes the step with the global sort
        atomicOr(&a.ctr->error, 16u);
        atomicOr(&a.ctr->abort, kAbortSort);
      }
    }
  } else if (tid == 0) {
    s_part[0] = 0;
    s_part[1] = a.n_coarse;
    s_misc[34] = 1;
  }
  if (tid == 0) {
    const unsigned long long base = atomicAdd(&a.ctr->sort_cursor, (unsigned long long)total);
    s_misc[36] = (uint32_t)base;
    s_misc[37] = (uint32_t)(base >> 32);
  }
  __syncthreads();
  const uint32_t np = s_misc[34];
  unsigned long long out = ((unsigned long long)s_misc[37] << 32) | s_misc[36];

  for (uint32_t p = 0; p < np; ++p) {
    const uint32_t c_lo = s_part[p], c_hi = s_part[p + 1];
    const uint64_t g_lo = (uint64_t)c_lo << a.gshift;
    const uint64_t span = (uint64_t)(c_hi - c_lo) << a.gshift;
    int fshift = 0;
    while ((span >> fshift) >= (uint64_t)kSortBins) ++fshift;
    for (int b = tid; b < kSortBins; b += kSortThreads) s_bins[b] = 0;
    if (tid == 0) {
      s_misc[32] = 0;
      s_misc[33] = 0;
    }
    __syncthreads();

    // ---- gather the part's anchors + fine histogram
    for (uint32_t r = wid; r < nr; r += kSortThreads / 32) {
      const RunRec run = run_at(r);
      for (uint32_t i0 = 0; i0 < run.count; i0 += 4 * 32) {  // a run is <= 128 hits: one trip,
        uint64_t kq[4];                                       // its eight loads in flight together
        float dq[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t i = i0 + u * 32 + lane;
          const bool has = i < run.count;
          kq[u] = has ? a.key_in[run.start + i] : ~0ull;
          dq[u] = has ? a.dist_in[run.start + i] : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (i0 + u * 32 >= run.count) break;
          const uint64_t k = kq[u];
          uint64_t g = 0;
          bool in = false;
          if (k != ~0ull) {
            g = coord(k);
            const uint32_t cb = (uint32_t)(g >> a.gshift);
            in = cb >= c_lo && cb < c_hi;
          }
          const unsigned m = __ballot_sync(full, in);
          if (!m) continue;
          uint32_t base = 0;
          if (lane == 0) base = atomicAdd(&s_misc[32], (uint32_t)__popc(m));
          base = __shfl_sync(full, base, 0);
          if (in) {
            const uint32_t slot = base + __popc(m & lt);
            if (slot < (uint32_t)kSortCap) {  // always true: part sizes are exact
              s_key[slot] = k;
              s_dist[slot] = dq[u];
              atomicAdd(&s_bins[(uint32_t)((g - g_lo) >> fshift)], 1u);
            }
          }
        }
      }
    }
    __syncthreads();
    const uint32_t n = min(s_misc[32], (uint32_t)kSortCap);

    // ---- exclusive scan of the fine histogram (8 consecutive bins per thread)
    {
      uint32_t v[kSortBins / kSortThreads], sum = 0;
#pragma unroll
      for (int j = 0; j < kSortBins / kSortThreads; ++j) {
        v[j] = s_bins[tid * (kSortBins / kSortThreads) + j];
        sum += v[j];
      }
      uint32_t incl = sum;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(full, incl, d);
        if (lane >= d) incl += t;
      }
      if (lane == 31) s_misc[wid] = incl;
      __syncthreads();
      if (wid == 0) {
        const uint32_t w = lane < kSortThreads / 32 ? s_misc[lane] : 0u;
        uint32_t in2 = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const uint32_t t = __shfl_up_sync(full, in2, d);
          if (lane >= d) in2 += t;
        }
        s_misc[lane] = in2 - w;
      }
      __syncthreads();
      uint32_t run_sum = s_misc[wid] + incl - sum;
#pragma unroll
      for (int j = 0; j < kSortBins / kSortThreads; ++j) {
        s_bins[tid * (kSortBins / kSortThreads) + j] = run_sum;
        run_sum += v[j];
      }
    }
    __syncthreads();

    // ---- counting-sort scatter of the slots; afterwards s_bins[b] = end of bin b
    for (uint32_t slot = tid; slot < n; slot += kSortThreads) {
      const uint32_t bin = (uint32_t)((coord(s_key[slot]) - g_lo) >> fshift);
      s_order[atomicAdd(&s_bins[bin], 1u)] = (uint16_t)slot;
    }
    __syncthreads();

    // ---- order every bin by the full key (bucket | target | query)
    for (int b = tid; b < kSortBins; b += kSortThreads) {
      const uint32_t lo = b ? s_bins[b - 1] : 0u, hi = s_bins[b];
      const uint32_t m = hi - lo;
      if (m < 2) continue;
      bool by_thread = m <= (uint32_t)kSmallBin;
      if (!by_thread) {
        const uint32_t at = atomicAdd(&s_misc[33], 1u);
        if (at < (uint32_t)kBigBinCap) s_big[at] = (uint32_t)b;
        else by_thread = true;  // queue full: slow but correct
      }
      if (by_thread) {
        for (uint32_t x = lo + 1; x < hi; ++x) {
          const uint16_t ox = s_order[x];
          const uint64_t kx = s_key[ox];
          uint32_t y = x;
          while (y > lo && s_key[s_order[y - 1]] > kx) {
            s_order[y] = s_order[y - 1];
            --y;
          }
          s_order[y] = ox;
        }
      }
    }
    __syncthreads();
    const uint32_t nbig = min(s_misc[33], (uint32_t)kBigBinCap);
    for (uint32_t bi = wid; bi < nbig; bi += kSortThreads / 32) {
      const uint32_t b = s_big[bi];
      const uint32_t lo = b ? s_bins[b - 1] : 0u, hi = s_bins[b];
      const uint32_t m = hi - lo;
      for (uint32_t x = lane; x < m; x += 32) {
        const uint16_t ox = s_order[lo + x];
        const uint64_t kx = s_key[ox];
        uint32_t rank = 0;
        for (uint32_t y = 0; y < m; ++y) {
          const uint64_t ky = s_key[s_order[lo + y]];
          rank += (ky < kx || (ky == kx && y < x)) ? 1u : 0u;
        }
        s_order2[lo + rank] = ox;
      }
      __syncwarp();
      for (uint32_t x = lane; x < m; x += 32) s_order[lo + x] = s_order2[lo + x];
    }
    __syncthreads();

    // ---- write the part back, sorted
    for (uint32_t pos = tid; pos < n; pos += kSortThreads) {
      const uint32_t slot = s_order[pos];
      a.key_out[out + pos] = s_key[slot];
      a.dist_out[out + pos] = s_dist[slot];
    }
    out += n;
    __syncthreads();
  }
}


// ---------------------------------------------------------------------------------------
// k_part_sort: the same sort when the producers (search flush, carry injection) have already
// routed every anchor to one of n_parts equal-width coordinate ranges of its entry ("parts",
// part_of(g)) and recorded one run list and one exact count per (entry, part).  One CTA per
// (entry, part): no coarse pass, nothing read twice, nothing filtered; output positions come
// from an exclusive scan of the counts, so the result is globally ordered by
// (entry, bucket, target, query).  Two 100 KB CTAs share an SM and cover each other's barriers.
//   gather   the part's anchors are addressed as one flat range [0, n) through the scanned run
//            counts: a warp takes four runs at a time, lanes the anchors of a run, slot = run
//            offset + i, no atomics; the loads of the four runs are in flight together
//   then     fine histogram -> scan -> counting-sort scatter -> per-bin order -> write-back,
//            as in k_seg_sort.
struct PartSortArgs {
  const uint64_t *key_in;
  const float *dist_in;
  uint64_t *key_out;
  float *dist_out;
  const RunRec *runs;           // [B * n_parts][runs_cap]
  const uint32_t *run_count;    // [B * n_parts]
  uint32_t runs_cap;            // run records per list
  const uint32_t *part_total;   // [B * n_parts] anchors of the part (<= CAP, checked by the host)
  const uint32_t *out_base;     // [B * n_parts] exclusive scan of part_total
  uint32_t n_parts;
  uint64_t span;                // coordinates per part (part boundaries are fuzzy by float rounding:
                                // the fine bins clamp, which keeps them monotone in g)
  KeyLayout kl;
  const uint64_t *bucket_base;
  uint32_t n_buckets;
  Counters *ctr;                // error bit 4: a sub-range of an oversize part overflowed
};

constexpr size_t part_sort_smem_bytes(int cap, int bins) {
  return (size_t)cap * (8 + 4 + 2 + 2) + (size_t)bins * 4 + (size_t)(kRunsCap + 8) * 8 + (size_t)kBigBinCap * 4 + 64 * 4;
}

// largest anchor count of any (entry, part): the host picks the sort kernel with it
__global__ void k_max_u32(const uint32_t *__restrict__ v, size_t n, unsigned int *__restrict__ out) {
  uint32_t m = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    m = max(m, v[i]);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, d));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

template <int CAP, int THREADS, int BINS>
__global__ void __launch_bounds__(THREADS, THREADS >= 1024 ? 1 : (THREADS >= 512 ? 2 : 4)) k_part_sort(const PartSortArgs a) {
  static_assert(BINS % THREADS == 0, "bins per thread");
  static_assert(THREADS <= 1024 && THREADS % 32 == 0, "block shape");
  extern __shared__ __align__(16) unsigned char s_raw[];
  uint64_t *s_key = reinterpret_cast<uint64_t *>(s_raw);
  float *s_dist = reinterpret_cast<float *>(s_key + CAP);
  uint32_t *s_bins = reinterpret_cast<uint32_t *>(s_dist + CAP);
  uint32_t *s_run_start = s_bins + BINS;            // [kRunsCap + 8] one tile of the run list
  uint32_t *s_run_off = s_run_start + kRunsCap + 8;   // [kRunsCap + 8] exclusive scan of the run counts (+ end)
  uint32_t *s_big = s_run_off + kRunsCap + 8;       // [kBigBinCap]
  uint32_t *s_misc = s_big + kBigBinCap;            // [64]: 0..31 warp sums, 32 kept, 33 nbig, 34 tile base
  uint16_t *s_order = reinterpret_cast<uint16_t *>(s_misc + 64);
  uint16_t *s_order2 = s_order + CAP;

  const uint32_t idx = blockIdx.x;
  const uint32_t n_all = a.part_total[idx];
  if (n_all == 0 || a.ctr->abort) return;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const unsigned full = 0xffffffffu;
  const uint32_t nr = min(a.run_count[idx], a.runs_cap);
  const RunRec *runs = a.runs + (size_t)idx * a.runs_cap;
  const KeyLayout kl = a.kl;
  unsigned long long out = a.out_base[idx];
  const uint64_t g_part = (uint64_t)(idx % a.n_parts) * a.span;
  // A part that fits the CTA is sorted in one go (slot = position in the flat run range, no
  // filtering).  The rare oversize part is cut into n_sub coordinate sub-ranges sized for half
  // the capacity, each gathered by filtering the whole part; a sub-range that still overflows
  // raises error bit 4 and the host redoes the step's sort with the generic kernels.
  const uint32_t n_sub = n_all <= (uint32_t)CAP ? 1u : (2u * n_all + CAP - 1u) / (uint32_t)CAP;
  const uint64_t sub_span = (a.span + n_sub - 1) / n_sub;
  int fshift = 0;
  while ((sub_span >> fshift) >= (uint64_t)BINS) ++fshift;
  // bucket bases: from shared memory when the genome has <= 64 buckets (32 contigs x 2 strands)
  __shared__ uint64_t s_bb[64];
  const bool bb_local = a.n_buckets <= 64u;
  if (bb_local && tid < (int)a.n_buckets) s_bb[tid] = a.bucket_base[tid];
  auto coord = [&](uint64_t k) -> uint64_t {
    const uint32_t b = kl.bucket(k);
    return (bb_local ? s_bb[b] : __ldg(a.bucket_base + b)) + kl.target(k);
  };

  for (uint32_t sub = 0; sub < n_sub; ++sub) {
    const uint64_t g_lo = g_part + (uint64_t)sub * sub_span;
    // the first / last sub-range are open-ended: part boundaries are fuzzy (part_of)
    const uint64_t f_lo = sub == 0 ? 0ull : g_lo;
    const uint64_t f_hi = sub + 1 == n_sub ? ~0ull : g_lo + sub_span;
    for (int b = tid; b < BINS; b += THREADS) s_bins[b] = 0;
    if (tid == 0) {
      s_misc[32] = 0;
      s_misc[33] = 0;
      s_misc[34] = 0;
    }
    __syncthreads();

    // ---- gather + fine histogram: a warp takes four runs at a time, lanes the consecutive
    // anchors of a run (slot = run offset + i), all loads of the four runs in flight together
    auto place = [&](uint32_t h, uint64_t k, float d) {
      const uint64_t g = coord(k);
      uint32_t slot = h;
      if (n_sub > 1) slot = (g >= f_lo && g < f_hi) ? atomicAdd(&s_misc[32], 1u) : 0xFFFFFFFFu;
      if (slot < (uint32_t)CAP) {
        const uint32_t bin = g >= g_lo ? (uint32_t)min((g - g_lo) >> fshift, (uint64_t)(BINS - 1)) : 0u;
        s_key[slot] = k;
        s_dist[slot] = d;
        s_order2[slot] = (uint16_t)bin;  // kept for the scatter below
        atomicAdd(&s_bins[bin], 1u);
      }
    };
    // the run list goes through shared memory one tile of kRunsCap records at a time
    for (uint32_t t0 = 0; t0 < nr; t0 += (uint32_t)kRunsCap) {
      const uint32_t tn = min(nr - t0, (uint32_t)kRunsCap);
      const uint32_t tile_base = s_misc[34];  // anchors of the tiles before this one
      // ---- tile -> shared memory, exclusive scan of the counts (kPer consecutive runs a thread)
      {
        constexpr int kPer = (kRunsCap + THREADS - 1) / THREADS;
        uint32_t cnt[kPer], sum = 0;
#pragma unroll
        for (int j = 0; j < kPer; ++j) {
          const uint32_t r = (uint32_t)tid * kPer + j;
          RunRec rec = RunRec{0u, 0u};
          if (r < tn) rec = runs[t0 + r];
          if (r < (uint32_t)kRunsCap) s_run_start[r] = rec.start;
          cnt[j] = rec.count;
          sum += rec.count;
        }
        uint32_t incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const uint32_t t = __shfl_up_sync(full, incl, d);
          if (lane >= d) incl += t;
        }
        if (lane == 31) s_misc[wid] = incl;
        __syncthreads();
        uint32_t at = tile_base + incl - sum;
        for (int w = 0; w < wid; ++w) at += s_misc[w];
#pragma unroll
        for (int j = 0; j < kPer; ++j) {
          const uint32_t r = (uint32_t)tid * kPer + j;
          if (r < (uint32_t)kRunsCap) s_run_off[r] = at;
          at += cnt[j];
        }
        if (tid == THREADS - 1) {
          s_run_off[kRunsCap] = at;  // end of the tile = base of the next
        }
        __syncthreads();
      }
      const uint32_t tile_end = s_run_off[kRunsCap];
      // (a flat mapping -- 32 consecutive slots per warp, the run of each slot by binary search --
      // keeps every lane busy but measured slower: 89 against 76 ms per pass of config 2)
      for (uint32_t r0 = (uint32_t)wid * 4u; r0 < tn; r0 += (THREADS / 32) * 4u) {
        uint32_t st[4], of[4], cn[4];
        uint64_t kq[4];
        float dq[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t r = r0 + u;
          st[u] = 0;
          of[u] = 0;
          cn[u] = 0;
          if (r < tn) {
            st[u] = s_run_start[r];
            of[u] = s_run_off[r];
            cn[u] = (r + 1 < tn ? s_run_off[r + 1] : tile_end) - of[u];
          }
          kq[u] = ~0ull;
          dq[u] = 0.0f;
          if ((uint32_t)lane < cn[u]) {
            kq[u] = a.key_in[st[u] + lane];
            dq[u] = a.dist_in[st[u] + lane];
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if ((uint32_t)lane < cn[u]) place(of[u] + lane, kq[u], dq[u]);
          for (uint32_t i = 32u + lane; i < cn[u]; i += 32u)  // runs longer than a warp
            place(of[u] + i, a.key_in[st[u] + i], a.dist_in[st[u] + i]);
        }
      }
      __syncthreads();  // the tile's records are not needed any more
      if (tid == 0) s_misc[34] = tile_end;
      __syncthreads();
    }
    __syncthreads();
    uint32_t n = n_all;
    if (n_sub > 1) {
      n = s_misc[32];
      if (n > (uint32_t)CAP) {
        if (tid == 0) {
          atomicOr(&a.ctr->error, 16u);
          atomicOr(&a.ctr->abort, kAbortSort);
        }
        n = CAP;
      }
    }

    // ---- exclusive scan of the fine histogram (consecutive bins per thread)
    {
      uint32_t v[BINS / THREADS], sum = 0;
#pragma unroll
      for (int j = 0; j < BINS / THREADS; ++j) {
        v[j] = s_bins[tid * (BINS / THREADS) + j];
        sum += v[j];
      }
      uint32_t incl = sum;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(full, incl, d);
        if (lane >= d) incl += t;
      }
      if (lane == 31) s_misc[wid] = incl;
      __syncthreads();
      uint32_t wbase = 0;
      for (int w = 0; w < wid; ++w) wbase += s_misc[w];
      uint32_t run_sum = wbase + incl - sum;
#pragma unroll
      for (int j = 0; j < BINS / THREADS; ++j) {
        s_bins[tid * (BINS / THREADS) + j] = run_sum;
        run_sum += v[j];
      }
    }
    __syncthreads();

    // ---- counting-sort scatter of the slots; afterwards s_bins[b] = end of bin b
    for (uint32_t slot = tid; slot < n; slot += THREADS)
      s_order[atomicAdd(&s_bins[s_order2[slot]], 1u)] = (uint16_t)slot;
    __syncthreads();

    // ---- order every bin by the full key (bucket | target | query): every anchor counts the
    // mates of its bin with a smaller key (keys are unique), one anchor per thread and pass, so
    // all lanes work whatever the bin sizes are (58 % of the anchors share their bin with another
    // one at the usual fill; a thread-per-bin insertion sort left most lanes idle and the block
    // waiting for its densest bin).  The final order replaces the bin numbers in s_order2 once
    // every thread has read what it needs.
    {
      constexpr int kPer = (CAP + THREADS - 1) / THREADS;
      uint32_t placed[kPer];  // final position << 16 | slot
#pragma unroll
      for (int j = 0; j < kPer; ++j) {
        const uint32_t pos = (uint32_t)tid + (uint32_t)j * THREADS;
        placed[j] = 0xFFFFFFFFu;
        if (pos < n) {
          const uint32_t slot = s_order[pos];
          const uint32_t b = s_order2[slot];
          const uint32_t lo = b ? s_bins[b - 1] : 0u, hi = s_bins[b];
          uint32_t rank = 0;
          if (hi - lo > 1u) {
            const uint64_t kx = s_key[slot];
            for (uint32_t y = lo; y < hi; ++y) rank += s_key[s_order[y]] < kx ? 1u : 0u;
          }
          placed[j] = ((lo + rank) << 16) | slot;
        }
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < kPer; ++j)
        if (placed[j] != 0xFFFFFFFFu) s_order2[placed[j] >> 16] = (uint16_t)(placed[j] & 0xFFFFu);
    }
    __syncthreads();

    // ---- write the sub-range back, sorted
    for (uint32_t pos = tid; pos < n; pos += THREADS) {
      const uint32_t slot = s_order2[pos];
      a.key_out[out + pos] = s_key[slot];
      a.dist_out[out + pos] = s_dist[slot];
    }
    out += n;
    __syncthreads();
  }
}

}  // namespace sb
#endif
