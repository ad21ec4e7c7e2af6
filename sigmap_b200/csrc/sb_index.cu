// sb_index.cu -- index construction: every smb_index_* and smb_point_cloud_* entry point.  The
// point cloud built on the device from the sequences (k_cloud.cuh), and the device index
// (k_index_build.cuh) from a cloud wherever it comes from: every entry point uploads or builds its
// arrays, then runs cloud_extent and build_index_core.  DESIGN.md, "Device index build".
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <string>
#include <vector>

#include "k_cloud.cuh"
#include "k_index_build.cuh"
#include "sb_ctx.cuh"

namespace {

struct StageTimer {  // CUDA events between the stages of one build
  Event ev[9];
  int n = 0;
  cudaError_t mark(cudaStream_t s) {
    if (!ev[n]) {
      const cudaError_t e = cudaEventCreate(&ev[n].h);
      if (e != cudaSuccess) return e;
    }
    return cudaEventRecord(ev[n++], s);
  }
  double ms(int a, int b) const {
    float f = 0.0f;
    if (a < n && b < n) cudaEventElapsedTime(&f, ev[a], ev[b]);
    return f;
  }
};

constexpr size_t kCloudSlice = 16u << 20;  // bytes per pinned upload slice

}  // namespace

#define CLOUD_ALLOC(arr, k, what)                                                                             \
  do {                                                                                                        \
    if ((arr).alloc(k) != cudaSuccess)                                                                        \
      return fail(ctx, SMB_ERR_CAPACITY,                                                                      \
                  std::string("index build: out of device memory for ") + (what) + " (" +            \
                      std::to_string(((size_t)(k) * sizeof(*(arr).p)) >> 20) + " MiB more)");              \
  } while (0)

// What the KD-order build takes: device arrays plus the extent of the points the index sees.
struct IndexInput {
  const float *val;              // values the windows read (whole cloud, or a shard's runs)
  const uint64_t *pos;           // position of every window (whole cloud: of every point)
  const uint32_t *wsrc, *worig;  // shard: value index / whole-cloud index of each window (else null)
  uint64_t W;                    // windows, >= 1 (a rank that owns none passes one padding window)
  size_t n_points;               // points of the whole cloud
  float vmin, vmax;
  uint32_t max_tpos, max_bucket;
  std::vector<uint64_t> bucket_span;  // 1 + largest target per bucket (contig << 1 | strand)
};

// The KD-order build from device arrays, wherever they came from.  Window w starts at value
// wsrc[w] (w itself when wsrc is null: the whole cloud) and is point worig[w] of the whole cloud.
// A window table (wsrc) makes the index a contig shard.
static int build_index_core(smb_ctx *ctx, IndexInput &in) {
  const uint64_t W = in.W;
  const uint32_t n_leaves = (uint32_t)((W + kLeaf - 1) / kLeaf);
  const float vmin = in.vmin, span = std::max(in.vmax - in.vmin, 1e-6f);
  const std::vector<uint64_t> &bucket_span = in.bucket_span;
  const float *d_val = in.val;
  const uint64_t *d_pos = in.pos;
  const uint32_t *d_wsrc = in.wsrc, *d_worig = in.worig;
  cudaStream_t s = ctx->stream;
  DeviceIndex &di = ctx->index;
  di.sharded = false;
  DevBuf<uint64_t> code_a, code_b;
  DevBuf<uint32_t> w_a, w_b;
  DevBuf<unsigned char> tmp;
  DevBuf<uint32_t> ext_min, ext_max;
  const uint32_t *d_order = nullptr;  // null: the windows' own order (one leaf holds them all)
  if (W > (uint64_t)kLeaf) {
    // aligned KD order (k_index.cuh): one pass per power-of-two segment size, top down
    CK(code_a.ensure(W));
    CK(code_b.ensure(W));
    CK(w_a.ensure(W));
    CK(w_b.ensure(W));
    int log2s = 4;
    while ((1ull << log2s) < W) ++log2s;
    const unsigned blocks = (unsigned)((W + kKdThreads - 1) / kKdThreads);
    const size_t n_ext = (size_t)((W + 15) / 16) * kDim;
    CK(ext_min.ensure(n_ext));
    CK(ext_max.ensure(n_ext));
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, code_a.p, code_b.p, w_a.p, w_b.p, (uint64_t)W, 0, 64, s);
    CK(tmp.ensure(tb));
    uint32_t *ia = w_a.p, *ib = w_b.p;
    bool first = true;
    for (; log2s >= 4; --log2s) {
      const uint64_t n_seg = (W + (1ull << log2s) - 1) >> log2s;
      CK(cudaMemsetAsync(ext_min.p, 0xFF, n_seg * kDim * sizeof(uint32_t), s));
      CK(cudaMemsetAsync(ext_max.p, 0x00, n_seg * kDim * sizeof(uint32_t), s));
      k_kd_extent<<<blocks, kKdThreads, 0, s>>>(d_val, first ? nullptr : ia, d_wsrc, W, log2s, ext_min.p, ext_max.p);
      LAUNCH_CHECK();
      k_kd_keys<<<blocks, kKdThreads, 0, s>>>(d_val, first ? nullptr : ia, d_wsrc, W, log2s, ext_min.p, ext_max.p,
                                              code_a.p, ia);
      LAUNCH_CHECK();
      int seg_bits = 0;
      while ((1ull << seg_bits) < n_seg) ++seg_bits;
      CK(cub::DeviceRadixSort::SortPairs(tmp.p, tb, code_a.p, code_b.p, ia, ib, (uint64_t)W, 0, 32 + seg_bits, s));
      std::swap(ia, ib);
      first = false;
      ctx->stats.launches += 9;
    }
    d_order = ia;
  }
  CK(di.leaves.ensure((size_t)n_leaves * kLeafRec));
  CK(di.leaf_widx.ensure((size_t)n_leaves * kLeaf));
  k_build_leaves<<<(unsigned)(((uint64_t)n_leaves * kLeaf + 255) / 256), 256, 0, s>>>(
      d_val, d_pos, d_order, W, n_leaves, di.leaves.p, di.leaf_widx.p, d_wsrc, d_worig);
  LAUNCH_CHECK();
  IndexView ix{};
  ix.n_points = in.n_points;
  ix.n_windows = W;
  ix.n_leaves = n_leaves;
  ix.vmin = vmin;
  ix.inv_span = 1.0f / span;
  // level sizes bottom-up; storage top-down in one buffer, so the levels every query walks are a
  // prefix of it (staged in shared memory by the lean search kernel)
  int L = 0;
  for (uint32_t n_child = n_leaves;;) {
    if (L >= kMaxLevels) return fail(ctx, SMB_ERR_CAPACITY, "index hierarchy deeper than kMaxLevels");
    const uint32_t n_nodes = (n_child + kFan - 1) / kFan;
    if (n_nodes >= (1u << 28)) return fail(ctx, SMB_ERR_CAPACITY, "index level exceeds 2^28 nodes");
    ix.level_count[L++] = n_nodes;
    if (n_nodes <= (uint32_t)kFan) break;  // the search starts from all nodes of the top level
    n_child = n_nodes;
  }
  ix.n_levels = L;
  uint64_t total_rec = 0;
  ix.smem_from = L;
  ix.smem_bytes = 0;
  for (int l = L - 1; l >= 0; --l) {
    if (total_rec * kNodeRec > 0xFFFFFFF0ull) return fail(ctx, SMB_ERR_CAPACITY, "node levels exceed 2^32 records: shard the index");
    ix.level_off[l] = (uint32_t)(total_rec * kNodeRec);
    total_rec += ix.level_count[l];
    if (ix.smem_from == l + 1 && total_rec * kNodeRec * sizeof(uint2) <= kTopSmemMax) {
      ix.smem_from = l;
      ix.smem_bytes = (uint32_t)(total_rec * kNodeRec * sizeof(uint2));
    }
  }
  CK(di.nodes.ensure((size_t)total_rec * kNodeRec));
  for (int l = 0; l < L; ++l) {
    const uint32_t n_nodes = ix.level_count[l];
    const unsigned blocks = (unsigned)(((uint64_t)n_nodes * kFan + 255) / 256);
    if (l == 0)
      k_nodes_level0<<<blocks, 256, 0, s>>>(di.leaves.p, n_leaves, n_nodes, di.nodes.p + ix.level_off[0]);
    else
      k_nodes_up<<<blocks, 256, 0, s>>>(di.nodes.p + ix.level_off[l - 1], ix.level_count[l - 1], n_nodes,
                                        di.nodes.p + ix.level_off[l]);
    LAUNCH_CHECK();
  }
  ix.nodes = di.nodes.p;
  ix.leaves = di.leaves.p;
  ix.leaf_widx = di.leaf_widx.p;
  CK(cudaStreamSynchronize(s));
  {
    // linear coordinate g = bucket_base[bucket] + target: monotone in the sort order, dense
    // enough to be cut into equal-width bins by the per-entry sort
    std::vector<uint64_t> base(bucket_span.size() + 1, 0);
    for (size_t b = 0; b < bucket_span.size(); ++b) base[b + 1] = base[b] + bucket_span[b];
    CK(di.bucket_base.ensure(base.size()));
    CK(cudaMemcpy(di.bucket_base.p, base.data(), base.size() * sizeof(uint64_t), cudaMemcpyHostToDevice));
    di.g_total = base.back();
    di.gshift = 0;
    while ((base.back() >> di.gshift) >= (uint64_t)kCoarseBins) ++di.gshift;
    di.n_coarse = (uint32_t)(base.back() >> di.gshift) + 1;
  }
  di.ix = ix;
  di.max_tpos = in.max_tpos;
  di.max_bucket = in.max_bucket;
  di.sharded = in.wsrc != nullptr;
  index_installed(ctx);
  return SMB_OK;
}

// The whole cloud in device memory (*pos / *val, *count points).  Stage times go to
// ctx->build_stats (ms_index is left to the caller).
static int cloud_build(smb_ctx *ctx, const char *const *seqs, const uint32_t *lengths, uint32_t n,
                       const float *level_mean, DevBuf<uint64_t> &pos, DevBuf<float> &val, uint64_t *count) {
  using namespace cloud;
  if (n && (!seqs || !lengths)) return fail(ctx, SMB_ERR_ARG, "device index build: null sequences / lengths");
  if (!level_mean) return fail(ctx, SMB_ERR_ARG, "device index build: null level table");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  smb_build_stats &bs = ctx->build_stats;
  memset(&bs, 0, sizeof bs);
  bs.tile = ctx->cloud_tile;
  *count = 0;
  // segments: + strands by contig, then - strands (contigs under 11 bases have no window)
  std::vector<Seg> segs;
  std::vector<uint64_t> plus_off(n, 0);
  uint64_t n_bases = 0, n_pos = 0;
  for (uint32_t c = 0; c < n; ++c) {
    if (lengths[c] < (uint32_t)kMaskK) continue;
    if (!seqs[c]) return fail(ctx, SMB_ERR_ARG, "device index build: null sequence");
    plus_off[c] = n_bases;
    n_bases += lengths[c];
  }
  for (uint32_t strand = 0; strand < 2; ++strand)
    for (uint32_t c = 0; c < n; ++c) {
      if (lengths[c] < (uint32_t)kMaskK) continue;
      segs.push_back(Seg{plus_off[c], n_pos, lengths[c], c, strand, 0});
      n_pos += lengths[c] - kK + 1;
    }
  if (segs.empty()) {
    CLOUD_ALLOC(pos, 0, "the point cloud");
    CLOUD_ALLOC(val, 0, "the point cloud");
    return SMB_OK;
  }
  const uint32_t n_segs = (uint32_t)segs.size(), n_plus = n_segs / 2;
  bs.strands = n_segs;
  StageTimer tm;
  CK(tm.mark(s));
  // ---- upload the + strands through two pinned slices
  DevBuf<unsigned char> d_seq;
  CLOUD_ALLOC(d_seq, n_bases, "the reference sequences");
  {
    const size_t slice = kCloudSlice;
    Event done[2];
    if (!ctx->h_cloud_stage.p) CK(ctx->h_cloud_stage.alloc(2 * slice));
    CK(cudaEventCreateWithFlags(&done[0].h, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&done[1].h, cudaEventDisableTiming));
    int k = 0;
    cudaError_t e = cudaSuccess;
    for (uint32_t c = 0; c < n && e == cudaSuccess; ++c) {
      if (lengths[c] < (uint32_t)kMaskK) continue;
      for (uint64_t a = 0; a < lengths[c] && e == cudaSuccess; a += slice) {
        const size_t len = (size_t)std::min<uint64_t>(slice, lengths[c] - a);
        unsigned char *h = ctx->h_cloud_stage.p + (size_t)k * slice;
        if ((e = cudaEventSynchronize(done[k])) != cudaSuccess) break;
        memcpy(h, seqs[c] + a, len);
        if ((e = cudaMemcpyAsync(d_seq.p + plus_off[c] + a, h, len, cudaMemcpyHostToDevice, s)) != cudaSuccess) break;
        e = cudaEventRecord(done[k], s);
        k ^= 1;
      }
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return fail(ctx, SMB_ERR_CUDA, std::string("device index build: upload: ") + cudaGetErrorString(e));
  }
  ctx->stats.h2d_bytes += n_bases;
  DevBuf<Seg> d_segs;
  CLOUD_ALLOC(d_segs, n_segs, "the segment table");
  CK(cudaMemcpyAsync(d_segs.p, segs.data(), n_segs * sizeof(Seg), cudaMemcpyHostToDevice, s));
  CK(tm.mark(s));
  // ---- 11-mer census over the + strands
  std::vector<Chunk> chunks;
  for (uint32_t i = 0; i < n_plus; ++i)
    for (uint32_t p = 0; p < segs[i].len - kMaskK + 1; p += kChunkPos) chunks.push_back(Chunk{i, p});
  const size_t n_census = chunks.size();
  for (uint32_t i = 0; i < n_segs; ++i)
    for (uint32_t p = 0; p < segs[i].len - kK + 1; p += kChunkPos) chunks.push_back(Chunk{i, p});
  DevBuf<Chunk> d_chunks;
  DevBuf<uint32_t> d_hist;
  DevBuf<unsigned long long> d_total;
  CLOUD_ALLOC(d_chunks, chunks.size(), "the chunk table");
  CLOUD_ALLOC(d_hist, (size_t)1 << (2 * kMaskK), "the 11-mer histogram");
  CLOUD_ALLOC(d_total, 1, "the 11-mer histogram");
  CK(cudaMemcpyAsync(d_chunks.p, chunks.data(), chunks.size() * sizeof(Chunk), cudaMemcpyHostToDevice, s));
  CK(cudaMemsetAsync(d_hist.p, 0, d_hist.cap * sizeof(uint32_t), s));
  CK(cudaMemsetAsync(d_total.p, 0, sizeof(unsigned long long), s));
  k_cloud_census<<<(unsigned)n_census, 256, 0, s>>>(d_seq.p, d_segs.p, d_chunks.p, d_hist.p, d_total.p);
  LAUNCH_CHECK();
  CK(tm.mark(s));
  // ---- level hashes and mask, both strands
  DevBuf<uint16_t> d_hm;
  CLOUD_ALLOC(d_hm, n_pos, "the per-position level hashes");
  k_cloud_hm<<<(unsigned)(chunks.size() - n_census), 256, 0, s>>>(d_seq.p, d_segs.p, d_chunks.p + n_census, d_hist.p,
                                                                   d_total.p, d_hm.p);
  LAUNCH_CHECK();
  CK(tm.mark(s));
  CK(cudaStreamSynchronize(s));
  d_seq.release();
  d_hist.release();
  d_chunks.release();
  // ---- z-normalisation: sequential double sums per strand -> z table per segment
  DevBuf<float> d_lv, d_ztab;
  CLOUD_ALLOC(d_lv, kTable, "the level table");
  CLOUD_ALLOC(d_ztab, (size_t)n_segs * kTable, "the z tables");
  CK(cudaMemcpyAsync(d_lv.p, level_mean, kTable * sizeof(float), cudaMemcpyHostToDevice, s));
  // the mean as an exact integer sum in units of the smallest ulp of the table (k_cloud_zsums):
  // possible when every level is finite and a strand's sum of |level| / unit stays in an int64
  int unit_exp = 0, int_ok = 1;
  {
    int lo = 1 << 30;
    double q_max = 0.0;
    for (int i = 0; i < kTable; ++i) {
      const float x = level_mean[i];
      if (!std::isfinite(x)) int_ok = 0;
      else if (x != 0.0f) lo = std::min(lo, std::max(std::ilogb(x), -126) - 23);
    }
    if (lo == 1 << 30) lo = 0;
    for (int i = 0; i < kTable && int_ok; ++i) q_max = std::max(q_max, std::ldexp(std::fabs((double)level_mean[i]), -lo));
    uint32_t max_len = 0;
    for (const Seg &g : segs) max_len = std::max(max_len, g.len);
    if (!int_ok || q_max * (double)max_len >= 9.0e18) int_ok = 0;
    unit_exp = lo;
  }
  DevBuf<unsigned int> d_serial;
  CLOUD_ALLOC(d_serial, 1, "the z sums");
  CK(cudaMemsetAsync(d_serial.p, 0, sizeof(unsigned int), s));
  k_cloud_zsums<<<(n_segs + kZWarps - 1) / kZWarps, kZWarps * 32, 0, s>>>(d_segs.p, n_segs, d_hm.p, d_lv.p, int_ok,
                                                                           unit_exp, d_ztab.p, d_serial.p);
  LAUNCH_CHECK();
  CK(cudaMemcpyAsync(&bs.strands_serial_mean, d_serial.p, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
  CK(tm.mark(s));
  // ---- point selection: speculative tiles, fix-up, chain
  std::vector<Tile> tiles;
  const uint32_t T = std::max<uint32_t>(ctx->cloud_tile, 1);
  uint64_t n_tiles64 = 0;
  for (const Seg &g : segs) n_tiles64 += (g.len - kMaskK + 1 + (uint64_t)T - 1) / T;
  if (n_tiles64 >= 0xFFFFFFFFull) return fail(ctx, SMB_ERR_ARG, "device index build: more than 2^32 tiles: raise cloud_tile");
  tiles.reserve(n_tiles64);
  for (uint32_t i = 0; i < n_segs; ++i) {
    const uint32_t nw = segs[i].len - kMaskK + 1;
    for (uint32_t p = 0; p < nw; p += std::min(T, nw - p)) tiles.push_back(Tile{i, p, p + std::min(T, nw - p), 0});
  }
  const uint32_t n_tiles = (uint32_t)tiles.size();
  DevBuf<Tile> d_tiles;
  DevBuf<TileState> d_ts;
  DevBuf<uint8_t> d_flags;
  DevBuf<ChainStats> d_cs;
  DevBuf<unsigned long long> d_cnt, d_off;
  CLOUD_ALLOC(d_tiles, n_tiles, "the tile table");
  CLOUD_ALLOC(d_ts, n_tiles, "the tile states");
  CLOUD_ALLOC(d_flags, n_pos, "the keep flags");
  CLOUD_ALLOC(d_cs, 1, "the tile states");
  CLOUD_ALLOC(d_cnt, n_tiles, "the tile counts");
  CLOUD_ALLOC(d_off, n_tiles, "the tile counts");
  CK(cudaMemcpyAsync(d_tiles.p, tiles.data(), n_tiles * sizeof(Tile), cudaMemcpyHostToDevice, s));
  const unsigned tb = 128, tg = (n_tiles + tb - 1) / tb;
  k_cloud_spec<<<tg, tb, 0, s>>>(d_segs.p, d_tiles.p, n_tiles, d_hm.p, d_ztab.p, d_flags.p, d_ts.p);
  LAUNCH_CHECK();
  k_cloud_assume<<<1, 1, 0, s>>>(d_ts.p, n_tiles);
  LAUNCH_CHECK();
  k_cloud_fix<<<tg, tb, 0, s>>>(d_segs.p, d_tiles.p, n_tiles, d_hm.p, d_ztab.p, d_flags.p, d_ts.p);
  LAUNCH_CHECK();
  k_cloud_chain<<<1, 1, 0, s>>>(d_segs.p, d_tiles.p, n_tiles, d_hm.p, d_ztab.p, d_flags.p, d_ts.p, d_cs.p);
  LAUNCH_CHECK();
  k_cloud_counts<<<tg, tb, 0, s>>>(d_ts.p, n_tiles, d_cnt.p);
  LAUNCH_CHECK();
  {
    size_t tmp_bytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_cnt.p, d_off.p, (int64_t)n_tiles, s));
    DevBuf<unsigned char> tmp;
    CLOUD_ALLOC(tmp, tmp_bytes, "the tile scan");
    CK(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, d_cnt.p, d_off.p, (int64_t)n_tiles, s));
    ctx->stats.launches += 2;
    unsigned long long last_off = 0, last_cnt = 0;
    ChainStats cs{};
    CK(cudaMemcpyAsync(&last_off, d_off.p + n_tiles - 1, sizeof last_off, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(&last_cnt, d_cnt.p + n_tiles - 1, sizeof last_cnt, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(&cs, d_cs.p, sizeof cs, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    *count = last_off + last_cnt;
    bs.tiles = n_tiles;
    bs.tiles_rewalked = cs.rewalked;
    bs.tiles_unconverged = cs.unconverged;
    bs.tiles_redone = cs.redone;
  }
  CK(tm.mark(s));
  // ---- scatter
  CLOUD_ALLOC(pos, *count, "the point cloud");
  CLOUD_ALLOC(val, *count, "the point cloud");
  k_cloud_scatter<<<(unsigned)(((uint64_t)n_tiles * 32 + 255) / 256), 256, 0, s>>>(d_segs.p, d_tiles.p, n_tiles, d_hm.p,
                                                                                     d_ztab.p, d_flags.p, d_off.p, pos.p, val.p);
  LAUNCH_CHECK();
  CK(tm.mark(s));
  CK(cudaStreamSynchronize(s));
  bs.points = *count;
  bs.ms_upload = tm.ms(0, 1);
  bs.ms_census = tm.ms(1, 2);
  bs.ms_levels = tm.ms(2, 3);
  bs.ms_zsums = tm.ms(3, 4);
  bs.ms_select = tm.ms(4, 5);
  bs.ms_scatter = tm.ms(5, 6);
  return SMB_OK;
}

namespace {
struct DevPart {  // one rank's part of the cloud in device memory (host_index.cc PartSink)
  DevBuf<uint64_t> pos, run_off, run_first, w_pos;
  DevBuf<float> val;
  DevBuf<uint8_t> own;
  DevBuf<uint32_t> w_src, w_orig;
  uint64_t n_values = 0, n_runs = 0, n_windows = 0;
};
}  // namespace

// The rank's part of the device cloud; with windows, also the window table of its shard.
static int part_build(smb_ctx *ctx, const DevBuf<uint64_t> &pos, const DevBuf<float> &val, uint64_t n,
                      const uint32_t *owner, uint32_t n_contigs, uint32_t rank, bool windows, DevPart &out) {
  using namespace cloud;
  cudaStream_t s = ctx->stream;
  DevBuf<uint32_t> d_owner;
  CLOUD_ALLOC(d_owner, n_contigs, "the owner table");
  CK(cudaMemcpyAsync(d_owner.p, owner, n_contigs * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
  const uint64_t nb64 = (n + kPartBlock - 1) / kPartBlock;
  if (nb64 >= 0x7FFFFFFFull) return fail(ctx, SMB_ERR_CAPACITY, "device index build: cloud too large for one part pass");
  const uint32_t nb = (uint32_t)std::max<uint64_t>(nb64, 1);
  DevBuf<unsigned long long> blk, cnt3, off3;
  CLOUD_ALLOC(blk, nb, "the part counters");
  CLOUD_ALLOC(cnt3, 3 * (size_t)nb, "the part counters");
  CLOUD_ALLOC(off3, 3 * (size_t)nb + 3, "the part counters");
  CK(cudaMemsetAsync(blk.p, 0, nb * sizeof(unsigned long long), s));
  if (n) {
    k_part_count<<<nb, kPartThreads, 0, s>>>(pos.p, n, d_owner.p, rank, blk.p);
    LAUNCH_CHECK();
  }
  k_part_unpack<<<(nb + 255) / 256, 256, 0, s>>>(blk.p, nb, cnt3.p);
  LAUNCH_CHECK();
  size_t tmp_bytes = 0;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, cnt3.p, off3.p, (int64_t)nb, s));
  DevBuf<unsigned char> tmp;
  CLOUD_ALLOC(tmp, tmp_bytes, "the part scan");
  for (int k = 0; k < 3; ++k)
    CK(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, cnt3.p + (size_t)k * nb, off3.p + (size_t)k * nb, (int64_t)nb, s));
  ctx->stats.launches += 3;
  unsigned long long last[6];
  for (int k = 0; k < 3; ++k) {
    CK(cudaMemcpyAsync(last + 2 * k, off3.p + (size_t)k * nb + nb - 1, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(last + 2 * k + 1, cnt3.p + (size_t)k * nb + nb - 1, 8, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  out.n_values = last[0] + last[1];
  out.n_runs = last[2] + last[3];
  out.n_windows = last[4] + last[5];
  CLOUD_ALLOC(out.pos, out.n_values, "the rank's part");
  CLOUD_ALLOC(out.val, out.n_values, "the rank's part");
  CLOUD_ALLOC(out.own, out.n_values, "the rank's part");
  CLOUD_ALLOC(out.run_off, out.n_runs + 1, "the rank's part");
  CLOUD_ALLOC(out.run_first, out.n_runs, "the rank's part");
  if (windows) {
    CLOUD_ALLOC(out.w_pos, out.n_windows, "the shard's windows");
    CLOUD_ALLOC(out.w_src, out.n_windows, "the shard's windows");
    CLOUD_ALLOC(out.w_orig, out.n_windows, "the shard's windows");
  }
  if (n) {
    k_part_emit<<<nb, kPartThreads, 0, s>>>(pos.p, val.p, n, d_owner.p, rank, off3.p, nb, out.pos.p, out.val.p,
                                            out.own.p, out.run_off.p, out.run_first.p, windows ? out.w_pos.p : nullptr,
                                            out.w_src.p, out.w_orig.p);
    LAUNCH_CHECK();
  }
  const uint64_t end = out.n_values;
  CK(cudaMemcpyAsync(out.run_off.p + out.n_runs, &end, sizeof end, cudaMemcpyHostToDevice, s));
  CK(cudaStreamSynchronize(s));
  return SMB_OK;
}

constexpr uint32_t kAnyContig = 0xFFFFFFFFu;

// vmin / vmax, the largest target and the bucket spans of the n points (pos, val) the index sees.
// The points each entry point passes, and the bucket table it gets:
//   smb_index_set_points, smb_index_load,    the whole cloud      up to the largest bucket seen
//   smb_index_build without owner
//   smb_index_set_points_sharded             the whole cloud      up to the largest bucket seen
//   smb_index_set_points_part,               the part's values    all 2 * contig_limit buckets (every
//   smb_index_build with owner                                    rank numbers the buckets alike)
// A point on a contig >= contig_limit is an error: part_build indexes the owner table by contig.
static int cloud_extent(smb_ctx *ctx, const uint64_t *pos, const float *val, uint64_t n, uint32_t contig_limit,
                        bool all_buckets, IndexInput &in) {
  using namespace cloud;
  cudaStream_t s = ctx->stream;
  DevBuf<CloudExtent> d_ext;
  CLOUD_ALLOC(d_ext, 1, "the cloud extent");
  const CloudExtent init{0xFFFFFFFFu, 0u, 0u, 0u};
  CK(cudaMemcpyAsync(d_ext.p, &init, sizeof init, cudaMemcpyHostToDevice, s));
  const unsigned grid = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->n_sm * 8);
  if (n) {
    k_cloud_extent<<<grid, 256, 0, s>>>(pos, val, n, d_ext.p);
    LAUNCH_CHECK();
  }
  CloudExtent ext{};
  CK(cudaMemcpyAsync(&ext, d_ext.p, sizeof ext, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (n && (ext.max_bucket >> 1) >= contig_limit)
    return fail(ctx, SMB_ERR_ARG, "point cloud names a contig beyond n_contigs");
  const size_t n_buckets = all_buckets ? 2 * (size_t)contig_limit : (n ? (size_t)ext.max_bucket + 1 : 0);
  DevBuf<unsigned long long> d_span;
  CLOUD_ALLOC(d_span, n_buckets, "the cloud extent");
  CK(cudaMemsetAsync(d_span.p, 0, n_buckets * sizeof(unsigned long long), s));
  if (n) {
    k_bucket_span<<<grid, 256, 0, s>>>(pos, n, d_span.p);
    LAUNCH_CHECK();
  }
  in.bucket_span.resize(n_buckets);
  CK(cudaMemcpyAsync(in.bucket_span.data(), d_span.p, n_buckets * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  in.vmin = n ? ord2f(ext.vmin_ord) : 0.0f;
  in.vmax = n ? ord2f(ext.vmax_ord) : 0.0f;
  in.max_tpos = ext.max_tpos;
  in.max_bucket = all_buckets ? (uint32_t)n_buckets - 1u : ext.max_bucket;
  return SMB_OK;
}

template <class T>
static int upload(smb_ctx *ctx, DevBuf<T> &d, const T *h, size_t n, const char *what) {
  CLOUD_ALLOC(d, n, what);
  CK(cudaMemcpyAsync(d.p, h, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return SMB_OK;
}

// The unsharded index over the whole cloud (N points in device memory).
static int build_whole(smb_ctx *ctx, const uint64_t *pos, const float *val, uint64_t N) {
  if (N < (uint64_t)kDim) return fail(ctx, SMB_ERR_ARG, "point cloud smaller than the index dimension");
  const uint64_t W = N - (kDim - 1);
  if (W > 0xFFFFFFF0ull) return fail(ctx, SMB_ERR_CAPACITY, "more than 2^32 window points: shard the index by contig");
  IndexInput in{val, pos, nullptr, nullptr, W, (size_t)N, 0.0f, 0.0f, 0u, 0u, {}};
  const int rc = cloud_extent(ctx, pos, val, N, kAnyContig, false, in);
  return rc ? rc : build_index_core(ctx, in);
}

// A contig shard from the window table of `part` and the extent in `in`.  A rank that owns no
// contig (more ranks than contigs) keeps one padding window: its values are never inside any
// ball and its leaf carries no target.
static int build_shard(smb_ctx *ctx, DevPart &part, IndexInput &in) {
  if (in.n_points < (size_t)kDim) return fail(ctx, SMB_ERR_ARG, "point cloud smaller than the index dimension");
  if (part.n_values > 0xFFFFFFF0ull)
    return fail(ctx, SMB_ERR_CAPACITY, "more than 2^32 window points on one shard: use more ranks");
  if (part.n_windows == 0) {
    const float pad[kDim] = {kPadValue, kPadValue, kPadValue, kPadValue, kPadValue, kPadValue};
    const uint64_t pad_pos = ~0ull;
    const uint32_t zero = 0, none = 0xFFFFFFFFu;
    int rc;
    if ((rc = upload(ctx, part.val, pad, kDim, "the padding window")) ||
        (rc = upload(ctx, part.w_pos, &pad_pos, 1, "the padding window")) ||
        (rc = upload(ctx, part.w_src, &zero, 1, "the padding window")) ||
        (rc = upload(ctx, part.w_orig, &none, 1, "the padding window")))
      return rc;
    part.n_windows = 1;
  }
  in.val = part.val.p;
  in.pos = part.w_pos.p;
  in.wsrc = part.w_src.p;
  in.worig = part.w_orig.p;
  in.W = part.n_windows;
  return build_index_core(ctx, in);
}

extern "C" {

int smb_index_set_points(smb_ctx *ctx, const uint64_t *pos, const float *val, size_t n) {
  CK(cudaSetDevice(ctx->device));
  DevBuf<uint64_t> d_pos;
  DevBuf<float> d_val;
  int rc;
  if ((rc = upload(ctx, d_pos, pos, n, "the point cloud")) || (rc = upload(ctx, d_val, val, n, "the point cloud")))
    return rc;
  return build_whole(ctx, d_pos.p, d_val.p, n);
}

int smb_index_load(smb_ctx *ctx, const char *prefix) {
  uint64_t *pos = nullptr;
  float *val = nullptr;
  size_t n = 0;
  int dim = 0, ml = 0;
  int rc = smbh_pt_read(prefix, &pos, &val, &n, &dim, &ml);
  if (rc) return fail(ctx, rc, std::string("cannot read ") + prefix + ".pt");
  if (dim != kDim) {
    smbh_free(pos);
    smbh_free(val);
    return fail(ctx, SMB_ERR_ARG, "index dimension is not 6");
  }
  rc = smb_index_set_points(ctx, pos, val, n);
  smbh_free(pos);
  smbh_free(val);
  return rc;
}

int smb_index_set_contigs(smb_ctx *ctx, const uint32_t *lengths, uint32_t n_contigs) {
  ctx->contig_len.assign(lengths, lengths + n_contigs);
  return SMB_OK;
}

// The whole cloud is uploaded (12 bytes per point, besides the shard) and the shard's windows are
// taken on the device, as smb_index_build does with an owner table.
int smb_index_set_points_sharded(smb_ctx *ctx, const uint64_t *pos, const float *val, size_t n,
                                 const uint32_t *contig_owner, uint32_t n_contigs) {
  CK(cudaSetDevice(ctx->device));
  if (!ctx->ex) return fail(ctx, SMB_ERR_STATE, "join a shard group first (smb_shard_local_group / smb_shard_nccl_init)");
  for (uint32_t c = 0; c < n_contigs; ++c)
    if (contig_owner[c] >= (uint32_t)ctx->ex->world) return fail(ctx, SMB_ERR_ARG, "contig owner out of range");
  DevBuf<uint64_t> d_pos;
  DevBuf<float> d_val;
  int rc;
  if ((rc = upload(ctx, d_pos, pos, n, "the point cloud")) || (rc = upload(ctx, d_val, val, n, "the point cloud")))
    return rc;
  IndexInput in{nullptr, nullptr, nullptr, nullptr, 0, n, 0.0f, 0.0f, 0u, 0u, {}};
  if ((rc = cloud_extent(ctx, d_pos.p, d_val.p, n, n_contigs, false, in))) return rc;
  DevPart part;
  if ((rc = part_build(ctx, d_pos, d_val, n, contig_owner, n_contigs, (uint32_t)ctx->ex->rank, true, part))) return rc;
  d_pos.release();
  d_val.release();
  return build_shard(ctx, part, in);
}

// The part comes from the host (smbh_build_point_cloud_part), so its window table is taken here: a
// window starts at every own point that has five more values after it in its run and is a window
// of the whole cloud (index < N - 5).
int smb_index_set_points_part(smb_ctx *ctx, const smbh_cloud_part *part, uint32_t n_contigs) {
  CK(cudaSetDevice(ctx->device));
  if (!ctx->ex) return fail(ctx, SMB_ERR_STATE, "join a shard group first (smb_shard_local_group / smb_shard_nccl_init)");
  if (!part || !n_contigs) return fail(ctx, SMB_ERR_ARG, "smb_index_set_points_part: no part / no contigs");
  const uint64_t N = part->n_points_total;
  std::vector<uint64_t> w_pos;
  std::vector<uint32_t> w_src, w_orig;
  for (size_t k = 0; k < part->n_runs; ++k) {
    const uint64_t a = part->run_off[k], b = part->run_off[k + 1];
    for (uint64_t i = a; i < b; ++i) {
      const uint64_t global = part->run_first[k] + (i - a);
      if (!part->own[i] || i + (kDim - 1) >= b || global + (kDim - 1) >= N) continue;
      w_pos.push_back(part->pos[i]);
      w_src.push_back((uint32_t)i);
      w_orig.push_back((uint32_t)global);
    }
  }
  DevPart dp;
  dp.n_values = part->n_values;
  dp.n_windows = w_pos.size();
  int rc;
  if ((rc = upload(ctx, dp.pos, part->pos, dp.n_values, "the rank's part")) ||
      (rc = upload(ctx, dp.val, part->val, dp.n_values, "the rank's part")) ||
      (rc = upload(ctx, dp.w_pos, w_pos.data(), dp.n_windows, "the shard's windows")) ||
      (rc = upload(ctx, dp.w_src, w_src.data(), dp.n_windows, "the shard's windows")) ||
      (rc = upload(ctx, dp.w_orig, w_orig.data(), dp.n_windows, "the shard's windows")))
    return rc;
  IndexInput in{nullptr, nullptr, nullptr, nullptr, 0, (size_t)N, 0.0f, 0.0f, 0u, 0u, {}};
  if ((rc = cloud_extent(ctx, dp.pos.p, dp.val.p, dp.n_values, n_contigs, true, in))) return rc;
  return build_shard(ctx, dp, in);
}

// Read-sharded runs (SURVEY.md 8e mode 1): the index is built once, on `root`, and travels to
// the other ranks of the group over NVLink (ncclBroadcast, or peer copies inside one process)
// instead of being rebuilt from the point cloud by every rank.  Collective: every rank of the
// group calls it; only the root needs an index (and contigs) beforehand.
int smb_index_broadcast(smb_ctx *ctx, int root) {
  CK(cudaSetDevice(ctx->device));
  if (!ctx->ex) return fail(ctx, SMB_ERR_STATE, "join a group first (smb_shard_local_group / smb_shard_nccl_init)");
  if (root < 0 || root >= ctx->ex->world) return fail(ctx, SMB_ERR_ARG, "bad root");
  const bool is_root = ctx->ex->rank == root;
  if (is_root && !ctx->has_index) return fail(ctx, SMB_ERR_STATE, "the root has no index to broadcast");
  cudaStream_t s = ctx->stream;
  DeviceIndex &di = ctx->index;
  // ---- header: the index's scalars (the view's pointers are the root's) and the contig count
  struct Header {
    IndexScalars index;
    uint32_t n_contigs;
  } h{};
  if (is_root) {
    h.index = di;
    h.n_contigs = (uint32_t)ctx->contig_len.size();
  }
  DevBuf<unsigned char> d_h;
  CK(d_h.ensure(sizeof(Header)));
  if (is_root) CK(cudaMemcpyAsync(d_h.p, &h, sizeof(Header), cudaMemcpyHostToDevice, s));
  int rc = ctx->ex->broadcast(d_h.p, sizeof(Header), root, s, ctx->err);
  if (rc) return rc;
  CK(cudaMemcpyAsync(&h, d_h.p, sizeof(Header), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  // ---- the arrays, in place in the receivers' own buffers
  const IndexView &ix = h.index.ix;
  uint64_t n_nodes_rec = 0;
  for (int l = 0; l < ix.n_levels; ++l) n_nodes_rec += (uint64_t)ix.level_count[l] * kNodeRec;
  const uint64_t n_leaf_rec = (uint64_t)ix.n_leaves * kLeafRec, n_widx = (uint64_t)ix.n_leaves * kLeaf;
  const uint64_t n_bucket_base = (uint64_t)h.index.max_bucket + 2;
  if (!is_root) {
    CK(di.nodes.ensure(n_nodes_rec));
    CK(di.leaves.ensure(n_leaf_rec));
    CK(di.leaf_widx.ensure(n_widx));
    CK(di.bucket_base.ensure(n_bucket_base));
  }
  DevBuf<uint32_t> d_len;
  CK(d_len.ensure(std::max<uint32_t>(h.n_contigs, 1)));
  if (is_root && h.n_contigs)
    CK(cudaMemcpyAsync(d_len.p, ctx->contig_len.data(), h.n_contigs * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
  if ((rc = ctx->ex->broadcast(di.nodes.p, n_nodes_rec * sizeof(uint2), root, s, ctx->err))) return rc;
  if ((rc = ctx->ex->broadcast(di.leaves.p, n_leaf_rec * sizeof(uint2), root, s, ctx->err))) return rc;
  if ((rc = ctx->ex->broadcast(di.leaf_widx.p, n_widx * sizeof(uint32_t), root, s, ctx->err))) return rc;
  if ((rc = ctx->ex->broadcast(di.bucket_base.p, n_bucket_base * sizeof(uint64_t), root, s, ctx->err))) return rc;
  if ((rc = ctx->ex->broadcast(d_len.p, std::max<uint32_t>(h.n_contigs, 1) * sizeof(uint32_t), root, s, ctx->err))) return rc;
  ctx->stats.exchanges += 6;
  if (!is_root) {
    ctx->contig_len.resize(h.n_contigs);
    if (h.n_contigs)
      CK(cudaMemcpyAsync(ctx->contig_len.data(), d_len.p, h.n_contigs * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    static_cast<IndexScalars &>(di) = h.index;
    di.ix.nodes = di.nodes.p;
    di.ix.leaves = di.leaves.p;
    di.ix.leaf_widx = di.leaf_widx.p;
    index_installed(ctx);
  }
  CK(cudaStreamSynchronize(s));
  di.sharded = false;
  return SMB_OK;
}

uint64_t smb_index_num_points(const smb_ctx *ctx) { return ctx->has_index ? ctx->index.ix.n_points : 0; }
uint32_t smb_index_num_contigs(const smb_ctx *ctx) { return (uint32_t)ctx->contig_len.size(); }

int smb_point_cloud_build(smb_ctx *ctx, const char *const *seqs, const uint32_t *lengths, uint32_t n,
                          const float *level_mean, uint64_t **pos, float **val, size_t *count) {
  if (!pos || !val || !count) return fail(ctx, SMB_ERR_ARG, "smb_point_cloud_build: null output");
  *pos = nullptr;
  *val = nullptr;
  *count = 0;
  DevBuf<uint64_t> d_pos;
  DevBuf<float> d_val;
  uint64_t c = 0;
  int rc = cloud_build(ctx, seqs, lengths, n, level_mean, d_pos, d_val, &c);
  if (rc) return rc;
  uint64_t *P = (uint64_t *)malloc(std::max<uint64_t>(c, 1) * sizeof(uint64_t));
  float *V = (float *)malloc(std::max<uint64_t>(c, 1) * sizeof(float));
  if (!P || !V) {
    free(P);
    free(V);
    return fail(ctx, SMB_ERR_IO, "smb_point_cloud_build: out of host memory");
  }
  cudaError_t e = cudaMemcpy(P, d_pos.p, c * sizeof(uint64_t), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(V, d_val.p, c * sizeof(float), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) {
    free(P);
    free(V);
    return fail(ctx, SMB_ERR_CUDA, std::string("smb_point_cloud_build: ") + cudaGetErrorString(e));
  }
  ctx->stats.d2h_bytes += c * 12;
  *pos = P;
  *val = V;
  *count = c;
  return SMB_OK;
}

int smb_point_cloud_build_part(smb_ctx *ctx, const char *const *seqs, const uint32_t *lengths, uint32_t n,
                               const float *level_mean, const uint32_t *owner, uint32_t rank, smbh_cloud_part *out) {
  if (!out) return fail(ctx, SMB_ERR_ARG, "smb_point_cloud_build_part: null output");
  memset(out, 0, sizeof *out);
  if (!owner) return fail(ctx, SMB_ERR_ARG, "smb_point_cloud_build_part: null owner table");
  DevPart part;
  {
    DevBuf<uint64_t> d_pos;
    DevBuf<float> d_val;
    uint64_t c = 0;
    int rc = cloud_build(ctx, seqs, lengths, n, level_mean, d_pos, d_val, &c);
    if (rc) return rc;
    rc = part_build(ctx, d_pos, d_val, c, owner, n, rank, false, part);
    if (rc) return rc;
    out->n_points_total = c;
  }
  out->n_values = part.n_values;
  out->n_runs = part.n_runs;
  auto take = [](const void *src, size_t bytes, cudaError_t &e) -> void * {
    void *p = malloc(bytes ? bytes : 1);
    if (p && bytes && e == cudaSuccess) e = cudaMemcpy(p, src, bytes, cudaMemcpyDeviceToHost);
    return p;
  };
  cudaError_t e = cudaSuccess;
  out->pos = (uint64_t *)take(part.pos.p, part.n_values * sizeof(uint64_t), e);
  out->val = (float *)take(part.val.p, part.n_values * sizeof(float), e);
  out->own = (uint8_t *)take(part.own.p, part.n_values, e);
  out->run_off = (uint64_t *)take(part.run_off.p, (part.n_runs + 1) * sizeof(uint64_t), e);
  out->run_first = (uint64_t *)take(part.run_first.p, part.n_runs * sizeof(uint64_t), e);
  if (!out->pos || !out->val || !out->own || !out->run_off || !out->run_first || e != cudaSuccess) {
    smbh_cloud_part_free(out);
    return e != cudaSuccess ? fail(ctx, SMB_ERR_CUDA, std::string("smb_point_cloud_build_part: ") + cudaGetErrorString(e))
                            : fail(ctx, SMB_ERR_IO, "smb_point_cloud_build_part: out of host memory");
  }
  return SMB_OK;
}

int smb_index_build(smb_ctx *ctx, const char *const *seqs, const uint32_t *lengths, uint32_t n,
                    const float *level_mean, const uint32_t *contig_owner) {
  CK(cudaSetDevice(ctx->device));
  if (contig_owner) {
    if (!ctx->ex) return fail(ctx, SMB_ERR_STATE, "join a shard group first (smb_shard_local_group / smb_shard_nccl_init)");
    if (!n) return fail(ctx, SMB_ERR_ARG, "smb_index_build: no contigs");
    for (uint32_t c = 0; c < n; ++c)
      if (contig_owner[c] >= (uint32_t)ctx->ex->world) return fail(ctx, SMB_ERR_ARG, "contig owner out of range");
  }
  DevBuf<uint64_t> d_pos;
  DevBuf<float> d_val;
  uint64_t N = 0;
  int rc = cloud_build(ctx, seqs, lengths, n, level_mean, d_pos, d_val, &N);
  if (rc) return rc;
  StageTimer tm;
  CK(tm.mark(ctx->stream));
  if (!contig_owner) {
    rc = build_whole(ctx, d_pos.p, d_val.p, N);
  } else {
    DevPart part;
    rc = part_build(ctx, d_pos, d_val, N, contig_owner, n, (uint32_t)ctx->ex->rank, true, part);
    if (rc) return rc;
    d_pos.release();  // the rank keeps its part only
    d_val.release();
    IndexInput in{nullptr, nullptr, nullptr, nullptr, 0, (size_t)N, 0.0f, 0.0f, 0u, 0u, {}};
    rc = cloud_extent(ctx, part.pos.p, part.val.p, part.n_values, n, true, in);
    if (!rc) rc = build_shard(ctx, part, in);
  }
  CK(tm.mark(ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->build_stats.ms_index = tm.ms(0, 1);
  return rc;
}

int smb_index_build_stats(smb_ctx *ctx, smb_build_stats *out) {
  if (!out) return fail(ctx, SMB_ERR_ARG, "smb_index_build_stats: null output");
  *out = ctx->build_stats;
  return SMB_OK;
}

}  // extern "C"
