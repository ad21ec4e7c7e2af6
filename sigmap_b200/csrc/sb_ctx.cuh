// sb_ctx.cuh -- the context behind the C ABI (smb_ctx), shared by the two translation units of
// the library: sb_engine.cu (the step, the read scheduler, streaming, stage hooks) and sb_index.cu
// (index construction).  Private: not part of include/sigmap_b200.h.
#ifndef SB_CTX_CUH
#define SB_CTX_CUH

#include <cuda_runtime.h>

#include <memory>
#include <string>
#include <vector>

#include "sb_device.cuh"
#include "sb_exchange.cuh"

namespace sb {
struct SegRec;  // k_chain.cuh
struct ChainTmp;
struct PickRec;
struct CandRec;

struct RoundInfo {
  uint32_t stop, num_events, n_chains;
};
}  // namespace sb

using namespace sb;

struct SlotSpace {
  uint32_t n_slots = 0;
  DevBuf<SlotState> slots;
  DevBuf<ChainRec> pool_chain[2];
  DevBuf<CarryAnchor> pool_anchor[2];
  std::vector<uint32_t> h_events, h_nchains;  // host mirror, refreshed every round
  uint32_t round = 0;
};

struct Workspace {
  // per-entry
  DevBuf<uint32_t> entry_slot, n_features, n_raw_events, n_queries, q_off, feat_row;
  // queries in Morton order (lean search kernel) and the ones it leaves to the general kernel
  DevBuf<uint32_t> qkey_a, qkey_b, qpay_a, qpay_b, ovf_list;
  DevBuf<uint2> entry_info;
  DevBuf<unsigned char> qsort_temp;
  // event lookahead block of the offline path: features of chunks [r0, r1) of the active reads
  // (two of them: the next block is computed on the event stream while this one is being mapped)
  DevBuf<float> feat_cache[2];
  DevBuf<uint32_t> nf_cache[2], nraw_cache[2];
  int cache_cur = 0;
  // chunk table of the lookahead blocks (the event stream's own copies)
  DevBuf<uint64_t> blk_chunk_start;
  DevBuf<float> blk_chunk_offset, blk_chunk_scale;
  DevBuf<uint8_t> absent;
  DevBuf<uint64_t> chunk_start;
  DevBuf<float> chunk_offset, chunk_scale;
  // events (transposed)
  DevBuf<float> ps, pss, t1, t2, means, features;
  // anchors
  DevBuf<uint64_t> key_a, key_b;
  DevBuf<float> dist_a, dist_b, score, coef;
  DevBuf<uint32_t> pred, link_list, link_count, pend_count, seg_qmin;
  DevBuf<uint16_t> pend_list;
  DevBuf<SegRec> seg;
  DevBuf<RunRec> runs;
  DevBuf<uint32_t> run_count, entry_total, part_base;
  DevBuf<unsigned char> cub_temp;
  DevBuf<ChainTmp> chain_tmp;
  DevBuf<PickRec> pick;
  DevBuf<float> seg_max;
  DevBuf<uint32_t> n_scratch;
  // contig-sharded runs (sb_exchange.cuh)
  DevBuf<CandRec> cand_list, cand_all;
  DevBuf<unsigned long long> cand_counts;
  DevBuf<double> ctl;
  DevBuf<uint32_t> tags;
  // round readback
  DevBuf<uint32_t> ids;
  DevBuf<RoundInfo> round_info;
};

// The installed device index.  The scalar part is a plain value: smb_index_broadcast sends it as
// it is, and a receiver points `ix` at its own copies of the buffers.
struct IndexScalars {
  IndexView ix{};
  uint32_t max_tpos = 0, max_bucket = 0;
  int gshift = 0;
  uint32_t n_coarse = 1;
  uint64_t g_total = 1;  // linear coordinates of the whole index (sum of the bucket spans)
  bool sharded = false;  // holds only this rank's contigs (a contig-sharded index)
};
struct DeviceIndex : IndexScalars {
  DevBuf<uint2> leaves;          // 256-byte leaf records (values + {target, bucket})
  DevBuf<uint2> nodes;           // every node level, top level first
  DevBuf<uint32_t> leaf_widx;
  DevBuf<uint64_t> bucket_base;  // linear coordinate of every bucket's target 0 (k_sort.cuh)
};

struct smb_ctx {
  int device = 0;
  Stream stream;
  std::string err;
  // index
  bool has_index = false;
  DeviceIndex index;
  unsigned search_grid_main = 148 * 4;   // general search kernel: every CTA that fits
  unsigned n_sm = 148;
  bool search_lean = true;        // SMB_SEARCH=general: every query through the general kernel
  uint32_t front_cap = 0;         // SMB_FRONT_CAP=n: frontier slots of the lean kernel (tests lower it; smb_create: kFrontCap)
  uint32_t runs_cap_min = 0;      // SMB_RUNS_CAP=n: run records per (entry, part) list (0 = from the estimate)
  int dp_passes = 0;              // SMB_DP_PASSES=n (smb_create: kDpFreePasses)
  int prep_rounds = 0;            // SMB_PREP_ROUNDS=n: settle rounds inside k_chain_prep (0 = none; smb_create: kPrepRounds)
  uint32_t dp_pass_max_entries = 0;  // SMB_DP_TILES=n: per-tile DP pass up to n chunks per step (0 = never;
                                     // smb_create: kDpPassMaxEntries)
  int pipeline_mode = 0;          // SMB_PIPELINE=auto|on|off: wave-pipelined ticks (see map_read_set)
  uint32_t cloud_tile = 16384;    // SMB_CLOUD_TILE=n: window starts per tile of the device cloud's point selection
  smb_build_stats build_stats{};  // the last device cloud build (smb_index_build_stats)
  PinnedBuf<unsigned char> h_cloud_stage;  // two upload slices of the device cloud build
  uint32_t sort_queries_min = 200000;  // SMB_SORT_QUERIES_MIN=n: batches with fewer queries keep their natural order
  unsigned dp_grid = 148 * 8;     // persistent DP grid: every block that fits on the device
  bool part_sort = true;          // SMB_SORT=entry: always the one-CTA-per-entry sort (k_seg_sort)
  bool seg_sort = true;           // per-entry shared-memory sort; SMB_SORT=global forces the radix sort
  Stream stream_cp;  // the slices of every mapping call (host input: copy + K1; otherwise K1) run here
  std::vector<Event> slice_events;
  size_t upload_slice_bytes = 64u << 20;  // SMB_UPLOAD_SLICE_MB=n
  PinnedBuf<uint32_t> h_kept_pinned;  // kept length of every read, written by the device
  Stream stream_ev;  // lookahead event blocks run here, next to the mapping rounds
  Event ev_blk_t0[2], ev_blk_t1[2];
  Event ev_cp[2];  // around a mapping call's slices on the copy stream (K1 time of resident / device input)
  bool ev_overlap = true;            // SMB_EVENTS_OVERLAP=0: compute every block when it is needed
  double ev_survival_hint = 0.0;     // share of reads that went past their first chunk in the last call
  uint32_t ev_warp_max = 2048;    // event batches up to this many chunks run warp-per-chunk in shared memory
                                  // (SMB_EVENTS=thread: never, =warp: always)
  std::vector<uint32_t> contig_len;
  // uploaded reads
  size_t n_reads = 0;
  // the read set came from smb_map_reads_device: its samples stayed in the caller's buffer, `raw`
  // does not hold them, and smb_map_uploaded has nothing to map
  bool device_input = false;
  Event ev_input;  // smb_map_reads_device: orders the context's streams after the caller's
  DevBuf<int16_t> raw, kept;
  // read_off of an upload (n + 1); for device input the n read starts, then the n read ends
  DevBuf<uint64_t> d_read_off, d_kept_off;
  DevBuf<float> d_dig, d_range, d_offset;
  DevBuf<uint32_t> d_kept_len;
  std::vector<uint64_t> h_kept_off;
  std::vector<uint32_t> h_kept_len;
  std::vector<float> h_offset, h_scale;
  std::vector<uint32_t> h_feat_row;
  // work
  Workspace ws;
  SlotSpace map_slots;
  DevBuf<Counters> d_ctr;
  PinnedBuf<Counters> h_ctr;
  Event ev[8];
  Event timer[2];
  smb_stats stats{};
  uint32_t max_batch_chunks = 32768;
  uint64_t max_batch_anchors = 640ull << 20;  // x 32 B of sort/DP buffers = 20 GB of the 180 GB HBM
  uint64_t last_cap = 0;
  double est_anchors_per_chunk = 20000.0;
  double est_queries_per_chunk = 260.0;
  double runs_scale = 1.0;          // raised when a step overflowed its run tables
  // contig-sharded index: the exchange backend (null = this context holds every contig)
  std::unique_ptr<Exchange> ex;
  std::shared_ptr<LocalGroup> local_group;
  PinnedBuf<double> h_ctl;  // 4 doubles
  bool group_at_limit = false;
  // streaming
  std::unique_ptr<SlotSpace> stream_slots;
  smb_params stream_params{};
  std::vector<std::vector<int16_t>> stream_pending;  // kept samples not yet forming a chunk
  std::vector<float> stream_offset, stream_scale;
  std::vector<uint32_t> stream_chunks, stream_kept;
  // raw values kept by the (30, 200) pA filter form an interval [lo, hi] per channel (the
  // conversion is monotone in the raw value); lo > hi: nothing kept; generic: test every sample
  std::vector<int32_t> stream_lo, stream_hi;
  std::vector<uint8_t> stream_generic;
  PinnedBuf<int16_t> h_stream_stage;  // this round's chunks, channel after channel
  DevBuf<int16_t> d_stream_stage;
};

#define CK(call)                                                                      \
  do {                                                                                \
    cudaError_t e_ = (call);                                                          \
    if (e_ != cudaSuccess) {                                                          \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                  \
      return SMB_ERR_CUDA;                                                            \
    }                                                                                 \
  } while (0)

#define LAUNCH_CHECK()                                                                \
  do {                                                                                \
    ctx->stats.launches++;                                                            \
    cudaError_t e_ = cudaGetLastError();                                              \
    if (e_ != cudaSuccess) {                                                          \
      ctx->err = std::string("kernel launch: ") + cudaGetErrorString(e_);             \
      return SMB_ERR_CUDA;                                                            \
    }                                                                                 \
  } while (0)

static inline int fail(smb_ctx *ctx, int code, const std::string &msg) {
  ctx->err = msg;
  // a failed member must not leave its in-process shard peers waiting at a rendezvous
  if (ctx->local_group) ctx->local_group->abort_all();
  return code;
}

// sb_engine.cu: marks ctx->index as installed and sizes the general search kernel's grid for it
void index_installed(smb_ctx *ctx);

#endif
