// k_cloud.cuh -- the point cloud of `sigmap -i` built on the device, bit for bit the cloud of
// build_cloud in host_index.cc (which stays the specification and the reference the tests compare with).
//
// Layout.  A segment is one strand of one contig with at least 11 bases, in cloud order: every +
// strand by contig, then every - strand.  Only the + strands are uploaded; a - strand base is
// read through the complement of the + strand (non-ACGT stays ambiguous).  Per position p of a
// segment (p < L = len - 5 expected levels) one u16 holds the 6-mer hash of its expected level and,
// for the window starts p < len - 10, the mask bit.  A strand's z-scores depend on the 6-mer only
// (z = (level - mean) / sd with the strand's mean and sd), so a 4096-entry table per segment turns
// a hash into the exact float the host computes.
//
// Stages:
//   k_cloud_census  canonical 11-mer histogram (u32[4^11], L2-resident) + total, + strands only
//   k_cloud_hm      per position: level hash (incl. the Q1 read-past-the-6-mer quirk) + mask bit
//   k_cloud_zsums   per segment, one warp: the sum of the levels (exact integer sum, or sequential
//                   doubles) and the sequential double sum of the squared deviations -> z table
//   k_cloud_spec    per tile: the `last kept value` walk, assuming the tile's first unmasked
//                   position is kept
//   k_cloud_assume / k_cloud_fix / k_cloud_chain   fix-up to the true incoming state (DESIGN.md)
//   k_cloud_scatter warp per tile: pos / val of the kept positions at the scanned tile offsets
// and, for one rank's part of a contig-sharded index, k_part_count / k_part_emit; for the index build
// of any cloud, k_cloud_extent / k_bucket_span.
#pragma once
#include <cstdint>

#include "sb_device.cuh"

namespace cloud {

constexpr int kK = 6;
constexpr int kMaskK = 11;
constexpr int kTable = 1 << (2 * kK);  // 4096 6-mers
constexpr uint16_t kMaskBit = 0x8000;
constexpr uint32_t kChunkPos = 8192;   // positions per block of the position-parallel kernels
constexpr int kZWarps = 4;             // segments per block of k_cloud_zsums
constexpr int kZBatch = 256;           // levels a warp stages before its lane 0 adds them in order

struct Seg {
  uint64_t seq_off;  // first base in the uploaded + strands
  uint64_t pos_off;  // first position in the per-position arrays (L = len - 5 of them)
  uint32_t len;      // bases of the contig
  uint32_t contig;
  uint32_t strand;
  uint32_t pad;
};
struct Chunk {  // kChunkPos positions [p0, p0 + kChunkPos) of segment `seg`
  uint32_t seg, p0;
};
struct Tile {  // window starts [p0, p1) of segment `seg`
  uint32_t seg, p0, p1, pad;
};
struct TileState {
  float spec_last;       // last kept value of the speculative walk
  float in_last;         // incoming state the fix-up pass assumed ...
  float out_last;        // ... and the outgoing state under that assumption
  uint32_t cnt_spec;     // points the speculative walk kept
  uint32_t cnt;          // points the tile keeps (under the assumed, finally the true, state)
  uint32_t fix_end;      // end of the prefix whose keep flags the fix-up rewrote
  uint8_t trans;         // no unmasked position: the state passes through
  uint8_t in_any, out_any;
  uint8_t conv;          // the re-walk met the speculative walk
  uint8_t rewalked;      // the re-walk decided at least one position differently
  uint8_t pad[3];
};
struct ChainStats {  // written by k_cloud_chain
  unsigned long long rewalked, unconverged, redone;
};

__device__ __forceinline__ int code_of(unsigned char c) {
  switch (c | 0x20) {  // either case; nothing else folds onto a/c/g/t
    case 'a': return 0;
    case 'c': return 1;
    case 'g': return 2;
    case 't': return 3;
    default: return -1;
  }
}

// base i of a segment, -1 where ambiguous; i == len is the terminating NUL (ambiguous)
__device__ __forceinline__ int seg_base(const unsigned char *seq, const Seg &s, uint32_t i) {
  if (i >= s.len) return -1;
  if (s.strand == 0) return code_of(seq[s.seq_off + i]);
  const int c = code_of(seq[s.seq_off + (s.len - 1 - i)]);
  return c < 0 ? -1 : 3 ^ c;
}

// canonical 11-mer starting at p of the segment, or -1 when one of its bases is ambiguous
__device__ __forceinline__ long long kmer11(const unsigned char *seq, const Seg &s, uint32_t p) {
  uint64_t fw = 0, rv = 0;
  for (int j = 0; j < kMaskK; ++j) {
    const int c = seg_base(seq, s, p + j);
    if (c < 0) return -1;
    fw = (fw << 2) | (uint64_t)c;
    rv |= (uint64_t)(3 ^ c) << (2 * j);
  }
  return (long long)(fw < rv ? fw : rv);
}

__global__ void k_cloud_census(const unsigned char *seq, const Seg *segs, const Chunk *chunks,
                               uint32_t *hist, unsigned long long *total) {
  const Chunk ch = chunks[blockIdx.x];
  const Seg s = segs[ch.seg];
  const uint32_t n_starts = s.len - kMaskK + 1;
  uint32_t mine = 0;
  for (uint32_t k = threadIdx.x; k < kChunkPos; k += blockDim.x) {
    const uint32_t p = ch.p0 + k;
    if (p >= n_starts) break;
    const long long m = kmer11(seq, s, p);
    if (m >= 0) {
      atomicAdd(hist + m, 1u);
      ++mine;
    }
  }
  for (int o = 16; o; o >>= 1) mine += __shfl_xor_sync(0xFFFFFFFFu, mine, o);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(total, (unsigned long long)mine);
}

// expected_levels' hash of position p: bases 0..5 at p = 0; for p >= 1 the seven bases p..p+6
// without base 6 (p <= 6) or without base p (p > 6), ambiguous bases and the NUL read as 'A'
__device__ __forceinline__ uint32_t level_hash(const unsigned char *seq, const Seg &s, uint32_t p) {
  uint32_t h = 0;
  if (p == 0) {
    for (uint32_t i = 0; i < (uint32_t)kK; ++i) {
      const int c = seg_base(seq, s, i);
      h = (h << 2) | (uint32_t)(c < 0 ? 0 : c);
    }
    return h;
  }
  const uint32_t skip = p <= 6 ? 6u : p;
  for (uint32_t i = p; i <= p + kK; ++i) {
    if (i == skip) continue;
    const int c = seg_base(seq, s, i);
    h = (h << 2) | (uint32_t)(c < 0 ? 0 : c);
  }
  return h;
}

__global__ void k_cloud_hm(const unsigned char *seq, const Seg *segs, const Chunk *chunks, const uint32_t *hist,
                           const unsigned long long *total, uint16_t *hm) {
  const Chunk ch = chunks[blockIdx.x];
  const Seg s = segs[ch.seg];
  const uint32_t L = s.len - kK + 1, n_starts = s.len - kMaskK + 1;
  const float tot = __ull2float_rn(*total);
  for (uint32_t k = threadIdx.x; k < kChunkPos; k += blockDim.x) {
    const uint32_t p = ch.p0 + k;
    if (p >= L) break;
    uint32_t v = level_hash(seq, s, p);
    if (p < n_starts) {
      const long long m = kmer11(seq, s, p);
      // host: M[p] = (float)H[k] / (float)total > 0.0002f for complete k-mers; 1 where the window
      // ending at an ambiguous base starts; 0 for the other incomplete windows
      const bool masked = m >= 0 ? __fdiv_rn(__uint2float_rn(hist[m]), tot) > 0.0002f
                                 : seg_base(seq, s, p + kMaskK - 1) < 0;
      if (masked) v |= kMaskBit;
    }
    hm[s.pos_off + p] = (uint16_t)v;
  }
}

// One warp per segment; znormalise's two sums are sequential doubles.
//   mean: every level is an integer multiple of `unit` (2^unit_exp, the smallest ulp in the level
//   table), so every partial sum of the host's loop is one too, and while sum |x| < 2^53 unit each
//   of them is a double and every addition exact: the sequential sum is the exact sum, taken here
//   as an integer (int_ok: the table allows it; the bound is checked per strand).  Otherwise, and
//   always for the squares, lane 0 adds the values in sequence order while the other lanes stage
//   them kZBatch at a time, the next batch's hashes already in flight.
__device__ __forceinline__ double zterm(float x, int pass, double mean) {
  if (pass == 0) return (double)x;
  const double d = __dsub_rn((double)x, mean);
  return __dmul_rn(d, d);
}

__device__ double serial_sum(const uint16_t *h, uint64_t L, const float *lv, double *buf, uint32_t lane, int pass,
                             double mean) {
  constexpr int kPer = kZBatch / 32;
  uint16_t nxt[kPer];
  for (int k = 0; k < kPer; ++k) nxt[k] = (uint64_t)(lane + 32 * k) < L ? h[lane + 32 * k] : 0;
  double sum = 0.0;
  for (uint64_t base = 0; base < L; base += kZBatch) {
    const uint32_t n = (uint32_t)(L - base < (uint64_t)kZBatch ? L - base : (uint64_t)kZBatch);
    for (int k = 0; k < kPer; ++k) buf[lane + 32 * k] = zterm(lv[nxt[k] & (kTable - 1)], pass, mean);
    __syncwarp();
    for (int k = 0; k < kPer; ++k) {
      const uint64_t i = base + kZBatch + lane + 32 * k;
      nxt[k] = i < L ? h[i] : 0;
    }
    if (lane == 0) {
      if (n == (uint32_t)kZBatch) {
#pragma unroll 16
        for (int j = 0; j < kZBatch; ++j) sum = __dadd_rn(sum, buf[j]);
      } else {
        for (uint32_t j = 0; j < n; ++j) sum = __dadd_rn(sum, buf[j]);
      }
    }
    __syncwarp();
  }
  return __shfl_sync(0xFFFFFFFFu, sum, 0);
}

__global__ void k_cloud_zsums(const Seg *segs, uint32_t n_segs, const uint16_t *hm, const float *level_mean,
                              int int_ok, int unit_exp, float *ztab, unsigned int *n_serial) {
  __shared__ float lv[kTable];
  __shared__ double buf[kZWarps][kZBatch];
  for (int i = threadIdx.x; i < kTable; i += blockDim.x) lv[i] = level_mean[i];
  __syncthreads();
  const uint32_t w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t si = blockIdx.x * kZWarps + w;
  if (si >= n_segs) return;
  const Seg s = segs[si];
  const uint64_t L = s.len - kK + 1;
  const uint16_t *h = hm + s.pos_off;
  double total = 0.0;
  bool exact = false;
  if (int_ok) {
    long long q_sum = 0;
    unsigned long long q_abs = 0;
    for (uint64_t i = lane; i < L; i += 32) {
      const long long q = __double2ll_rn(ldexp((double)lv[h[i] & (kTable - 1)], -unit_exp));
      q_sum += q;
      q_abs += (unsigned long long)(q < 0 ? -q : q);
    }
    for (int o = 16; o; o >>= 1) {
      q_sum += __shfl_xor_sync(0xFFFFFFFFu, q_sum, o);
      q_abs += __shfl_xor_sync(0xFFFFFFFFu, q_abs, o);
    }
    exact = q_abs < (1ull << 53);
    if (exact) total = ldexp((double)q_sum, unit_exp);
  }
  if (!exact) {
    total = serial_sum(h, L, lv, buf[w], lane, 0, 0.0);
    if (lane == 0) atomicAdd(n_serial, 1u);
  }
  const double mean = __ddiv_rn(total, (double)L);
  const double ss = serial_sum(h, L, lv, buf[w], lane, 1, mean);
  const double sd = __dsqrt_rn(__ddiv_rn(ss, (double)(L - 1)));
  for (int i = lane; i < kTable; i += 32)
    ztab[(size_t)si * kTable + i] = __double2float_rn(__ddiv_rn(__dsub_rn((double)lv[i], mean), sd));
}

__device__ __forceinline__ bool keep_point(uint32_t p, bool any, float z, float last) {
  return p == 0 || !any || fabs((double)__fsub_rn(z, last)) > 0.01;
}

// Pass 1: the walk of one tile as if its first unmasked position were kept.  flags: bit 0 = kept
// by this walk, bit 1 = kept in the cloud (the fix-up rewrites bit 1 only).
__global__ void k_cloud_spec(const Seg *segs, const Tile *tiles, uint32_t n_tiles, const uint16_t *hm,
                             const float *ztab, uint8_t *flags, TileState *ts) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  const Tile tl = tiles[t];
  const uint64_t off = segs[tl.seg].pos_off;
  const float *zt = ztab + (size_t)tl.seg * kTable;
  bool first = true;
  float last = 0.0f;
  uint32_t cnt = 0;
  for (uint32_t p = tl.p0; p < tl.p1; ++p) {
    const uint16_t v = hm[off + p];
    if (v & kMaskBit) {
      flags[off + p] = 0;
      continue;
    }
    const float z = zt[v & (kTable - 1)];
    const bool keep = first || keep_point(p, true, z, last);
    first = false;
    flags[off + p] = keep ? 3 : 0;
    if (keep) {
      last = z;
      ++cnt;
    }
  }
  TileState st{};
  st.spec_last = last;
  st.cnt_spec = st.cnt = cnt;
  st.trans = first;
  ts[t] = st;
}

// Re-walk a tile from the state (any, last) until it keeps a position the speculative walk also
// kept: from there on both walks are the same.  Rewrites bit 1 of the flags on the way.
struct FixResult {
  bool conv, rewalked;
  bool any;
  float last;
  uint32_t end;
  int64_t delta;  // points kept minus points the speculative walk kept, over the rewritten prefix
};
__device__ FixResult fix_walk(const Tile &tl, uint64_t off, const float *zt, const uint16_t *hm, uint8_t *flags,
                              bool any, float last) {
  FixResult r{false, false, any, last, tl.p1, 0};
  for (uint32_t p = tl.p0; p < tl.p1; ++p) {
    const uint16_t v = hm[off + p];
    if (v & kMaskBit) continue;
    const float z = zt[v & (kTable - 1)];
    const bool keep = keep_point(p, r.any, z, r.last);
    const uint8_t f = flags[off + p];
    const bool spec = f & 1;
    if (keep && spec) {
      r.conv = true;
      r.end = p;
      break;
    }
    r.rewalked = true;
    flags[off + p] = (uint8_t)((f & 1) | (keep ? 2 : 0));
    r.delta += (int)keep - (int)spec;
    if (keep) {
      r.any = true;
      r.last = z;
    }
  }
  return r;
}

// The state every tile would receive if all tiles before it met their speculative walk: the
// speculative outgoing state of the nearest earlier tile with an unmasked position.  One thread;
// it only reads two words per tile.
__global__ void k_cloud_assume(TileState *ts, uint32_t n_tiles) {
  bool any = false;
  float last = 0.0f;
  for (uint32_t t = 0; t < n_tiles; ++t) {
    ts[t].in_any = any;
    ts[t].in_last = last;
    if (!ts[t].trans) {
      any = true;
      last = ts[t].spec_last;
    }
  }
}

// Pass 2, every tile at once, from the assumed incoming state.
__global__ void k_cloud_fix(const Seg *segs, const Tile *tiles, uint32_t n_tiles, const uint16_t *hm,
                            const float *ztab, uint8_t *flags, TileState *ts) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  TileState st = ts[t];
  if (st.trans) return;
  const Tile tl = tiles[t];
  const FixResult r = fix_walk(tl, segs[tl.seg].pos_off, ztab + (size_t)tl.seg * kTable, hm, flags, st.in_any,
                               st.in_last);
  st.conv = r.conv;
  st.rewalked = r.rewalked;
  st.out_any = r.conv ? 1 : r.any;
  st.out_last = r.conv ? st.spec_last : r.last;
  st.fix_end = r.end;
  st.cnt = (uint32_t)((int64_t)st.cnt_spec + r.delta);
  ts[t] = st;
}

// The true state, tile after tile (one thread).  Where it equals the state k_cloud_fix assumed,
// that pass's result stands; otherwise (after a tile that never met its speculative walk: a
// stretch of equal z, for instance) the tile is restored to its speculative flags and re-walked
// here from the true state.  Exact whatever the length of such a stretch; only slower.
__global__ void k_cloud_chain(const Seg *segs, const Tile *tiles, uint32_t n_tiles, const uint16_t *hm,
                              const float *ztab, uint8_t *flags, TileState *ts, ChainStats *cs) {
  bool any = false;
  float last = 0.0f;
  ChainStats c{0, 0, 0};
  for (uint32_t t = 0; t < n_tiles; ++t) {
    TileState st = ts[t];
    if (st.trans) {
      ++c.unconverged;
      continue;
    }
    const bool same = any == (bool)st.in_any && (!any || __float_as_uint(last) == __float_as_uint(st.in_last));
    if (!same) {
      const Tile tl = tiles[t];
      const uint64_t off = segs[tl.seg].pos_off;
      for (uint32_t p = tl.p0; p < st.fix_end; ++p) flags[off + p] = (flags[off + p] & 1) ? 3 : 0;
      const FixResult r = fix_walk(tl, off, ztab + (size_t)tl.seg * kTable, hm, flags, any, last);
      st.conv = r.conv;
      st.rewalked = r.rewalked;
      st.out_any = r.conv ? 1 : r.any;
      st.out_last = r.conv ? st.spec_last : r.last;
      st.fix_end = r.end;
      st.cnt = (uint32_t)((int64_t)st.cnt_spec + r.delta);
      ts[t] = st;
      ++c.redone;
    }
    c.rewalked += st.rewalked;
    c.unconverged += !st.conv;
    any = st.out_any;
    last = st.out_last;
  }
  *cs = c;
}

__global__ void k_cloud_counts(const TileState *ts, uint32_t n_tiles, unsigned long long *cnt) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n_tiles) cnt[t] = ts[t].trans ? 0ull : ts[t].cnt;
}

// One warp per tile: 32 positions at a time, the kept ones compacted by ballot (coalesced writes).
__global__ void k_cloud_scatter(const Seg *segs, const Tile *tiles, uint32_t n_tiles, const uint16_t *hm,
                                const float *ztab, const uint8_t *flags, const unsigned long long *tile_off,
                                uint64_t *pos, float *val) {
  const uint32_t t = (uint32_t)(((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (t >= n_tiles) return;
  const Tile tl = tiles[t];
  const Seg s = segs[tl.seg];
  const float *zt = ztab + (size_t)tl.seg * kTable;
  uint64_t o = tile_off[t];
  for (uint32_t base = tl.p0; base < tl.p1; base += 32) {
    const uint32_t p = base + lane;
    const bool keep = p < tl.p1 && (flags[s.pos_off + p] & 2);
    const uint32_t mask = __ballot_sync(0xFFFFFFFFu, keep);
    if (keep) {
      const uint64_t at = o + __popc(mask & ((1u << lane) - 1));
      pos[at] = ((((uint64_t)s.contig << 32) | p) << 1) | (uint64_t)s.strand;
      val[at] = zt[hm[s.pos_off + p] & (kTable - 1)];
    }
    o += __popc(mask);
  }
}

// ---- one rank's part (host_index.cc PartSink): point i of the cloud is taken when its contig is
// the rank's or one of the five points before it is; a run starts at a taken point whose
// predecessor was not taken or was the fifth point after the last own one.  Windows start at own
// points i < n - 5.  Counts (taken, run starts, windows) are packed 21 bits each per block.
constexpr int kPartThreads = 256, kPartPer = 4, kPartBlock = kPartThreads * kPartPer;

__device__ __forceinline__ bool part_own(const uint64_t *pos, int64_t i, const uint32_t *owner, uint32_t rank) {
  return i >= 0 && owner[pos[i] >> 33] == rank;
}

__device__ __forceinline__ uint64_t part_flags(const uint64_t *pos, uint64_t n, uint64_t i, const uint32_t *owner,
                                               uint32_t rank, bool *own_out) {
  bool m[7];  // m[k] = point i - k is the rank's
  for (int k = 0; k < 7; ++k) m[k] = part_own(pos, (int64_t)i - k, owner, rank);
  const bool before = m[1] || m[2] || m[3] || m[4] || m[5];
  const bool taken = m[0] || before;
  const bool prev_taken = before || m[6];
  const bool prev_closed = !before && m[6];  // point i - 1 was the fifth after the last own one
  const bool start = taken && (i == 0 || !prev_taken || prev_closed);
  const bool window = m[0] && i + 5 < n;
  *own_out = m[0];
  return (uint64_t)taken | ((uint64_t)start << 21) | ((uint64_t)window << 42);
}

__global__ void k_part_count(const uint64_t *pos, uint64_t n, const uint32_t *owner, uint32_t rank,
                             unsigned long long *blk) {
  __shared__ unsigned long long s;
  if (threadIdx.x == 0) s = 0;
  __syncthreads();
  unsigned long long c = 0;
  for (int k = 0; k < kPartPer; ++k) {
    const uint64_t i = (uint64_t)blockIdx.x * kPartBlock + k * kPartThreads + threadIdx.x;
    bool own;
    if (i < n) c += part_flags(pos, n, i, owner, rank, &own);
  }
  atomicAdd(&s, c);
  __syncthreads();
  if (threadIdx.x == 0) blk[blockIdx.x] = s;
}

// blk_off: exclusive scan of the three packed counters, unpacked (3 x n_blocks u64)
__global__ void k_part_unpack(const unsigned long long *blk, uint32_t n_blocks, unsigned long long *cnt3) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_blocks) return;
  const unsigned long long v = blk[b], m = (1ull << 21) - 1;
  cnt3[b] = v & m;
  cnt3[n_blocks + b] = (v >> 21) & m;
  cnt3[2 * (size_t)n_blocks + b] = (v >> 42) & m;
}

// Writes the part (pos / val / own at the taken index; run_off / run_first per run) and, when
// w_pos is set, the window table the index build takes (window position, its value's index in
// the part, its index in the whole cloud).  Points are visited in order inside a block: the
// counters are scanned over the block's kPartBlock points.
__global__ void k_part_emit(const uint64_t *pos, const float *val, uint64_t n, const uint32_t *owner, uint32_t rank,
                            const unsigned long long *off3, uint32_t n_blocks, uint64_t *p_pos, float *p_val,
                            uint8_t *p_own, uint64_t *run_off, uint64_t *run_first, uint64_t *w_pos,
                            uint32_t *w_src, uint32_t *w_orig) {
  __shared__ unsigned long long wsum[kPartThreads / 32];
  const unsigned long long m21 = (1ull << 21) - 1;
  unsigned long long base[3] = {off3[blockIdx.x], off3[n_blocks + blockIdx.x], off3[2 * (size_t)n_blocks + blockIdx.x]};
  for (int k = 0; k < kPartPer; ++k) {
    const uint64_t i = (uint64_t)blockIdx.x * kPartBlock + k * kPartThreads + threadIdx.x;
    bool own = false;
    const unsigned long long f = i < n ? part_flags(pos, n, i, owner, rank, &own) : 0ull;
    // block-wide exclusive scan of the packed flags (warp scan + warp totals)
    const uint32_t lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned long long x = f;
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long y = __shfl_up_sync(0xFFFFFFFFu, x, o);
      if (lane >= (uint32_t)o) x += y;
    }
    if (lane == 31) wsum[w] = x;
    __syncthreads();
    unsigned long long before = x - f, total = 0;
    for (uint32_t j = 0; j < kPartThreads / 32; ++j) {
      if (j < w) before += wsum[j];
      total += wsum[j];
    }
    __syncthreads();
    const uint64_t ti = base[0] + (before & m21), ri = base[1] + ((before >> 21) & m21),
                   wi = base[2] + ((before >> 42) & m21);
    if (f & 1) {
      p_pos[ti] = pos[i];
      p_val[ti] = val[i];
      p_own[ti] = own;
    }
    if ((f >> 21) & 1) {
      run_off[ri] = ti;
      run_first[ri] = i;
    }
    if (((f >> 42) & 1) && w_pos) {
      w_pos[wi] = pos[i];
      w_src[wi] = (uint32_t)ti;
      w_orig[wi] = (uint32_t)i;
    }
    base[0] += total & m21;
    base[1] += (total >> 21) & m21;
    base[2] += (total >> 42) & m21;
  }
}

// What the index build needs besides the arrays themselves: vmin / vmax of the values, the
// largest target and the largest bucket (contig << 1 | strand) of the positions ...
struct CloudExtent {
  unsigned int vmin_ord, vmax_ord, max_tpos, max_bucket;
};
__global__ void k_cloud_extent(const uint64_t *pos, const float *val, uint64_t n, CloudExtent *ext) {
  unsigned int lo = 0xFFFFFFFFu, hi = 0, tp = 0, bk = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t o = sb::f2ord(val[i]);
    lo = min(lo, o);
    hi = max(hi, o);
    const uint64_t P = pos[i];
    tp = max(tp, (uint32_t)(P >> 1));
    bk = max(bk, (uint32_t)(((P >> 33) << 1) | (P & 1)));
  }
  for (int o = 16; o; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xFFFFFFFFu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xFFFFFFFFu, hi, o));
    tp = max(tp, __shfl_xor_sync(0xFFFFFFFFu, tp, o));
    bk = max(bk, __shfl_xor_sync(0xFFFFFFFFu, bk, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(&ext->vmin_ord, lo);
    atomicMax(&ext->vmax_ord, hi);
    atomicMax(&ext->max_tpos, tp);
    atomicMax(&ext->max_bucket, bk);
  }
}

// ... and 1 + the largest target of every bucket (the table has a slot for every bucket of the
// positions).  Each run of non-decreasing targets inside a bucket gives its last target, so any
// point order yields the exact maximum; a cloud ordered by bucket and target, as every cloud
// built by this library is, takes one atomic per bucket.
__global__ void k_bucket_span(const uint64_t *pos, uint64_t n, unsigned long long *bucket_span) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t P = pos[i];
    const uint32_t t = (uint32_t)(P >> 1), b = (uint32_t)(((P >> 33) << 1) | (P & 1));
    bool last = i + 1 == n;
    if (!last) {
      const uint64_t Q = pos[i + 1];
      last = (uint32_t)(((Q >> 33) << 1) | (Q & 1)) != b || (uint32_t)(Q >> 1) < t;
    }
    if (last) atomicMax(bucket_span + b, (unsigned long long)t + 1);
  }
}

}  // namespace cloud
