/*
 * sigmap_b200.h -- C ABI of the B200-native Sigmap mapping hot path.
 *
 * This is the drop-in boundary (SURVEY.md 8b): plain pointers and sizes, no C++ or torch
 * types, no exceptions, never exit().  Every call returns SMB_OK (0) or a negative
 * SMB_ERR_* code; smb_last_error(ctx) holds the message.  One context owns one GPU and
 * all device memory; calls on one context must be serialised by the caller.
 *
 * Each entry point names the reference interface it replaces (file:line are relative to
 * the reference repository haowenz/sigmap @ c9a4048).  INTEGRATION.md shows the binding
 * a maintainer of the reference would add.
 *
 * There is NO CPU fallback: without a CUDA device smb_create() fails and nothing else
 * can be called.  Host-only helpers (file formats, simulator) are prefixed smbh_.
 */
#ifndef SIGMAP_B200_H
#define SIGMAP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMB_OK 0
#define SMB_ERR_ARG (-1)      /* bad argument / call order */
#define SMB_ERR_IO (-2)       /* file missing or malformed */
#define SMB_ERR_CUDA (-3)     /* CUDA runtime error (message has the cudaError string) */
#define SMB_ERR_NO_DEVICE (-4)/* no usable CUDA device: the library refuses to run */
#define SMB_ERR_CAPACITY (-5) /* a bounded device buffer overflowed (message says which) */
#define SMB_ERR_STATE (-6)    /* e.g. mapping requested before an index was loaded */

#define SMB_CHUNK 4000        /* samples per chunk: sigmap.cc:639 */
#define SMB_DIM 6             /* index dimension: sigmap.cc:1422 */
#define SMB_MAX_HITS 5000     /* num_nearest_points: spatial_index.cc:290 */

typedef struct smb_ctx smb_ctx;
typedef struct smb_batch smb_batch;

/* Mapping knobs = the `Sigmap` mapping constructor arguments (sigmap.h:45-71) with the
 * CLI defaults of sigmap.cc:1380-1419. */
typedef struct smb_params {
  float search_radius;            /* --search-radius            0.08 (squared L2, Q4) */
  int32_t step_size;              /* --step-size                2    */
  int32_t max_num_chunks;         /* --max-num-chunks           30   */
  int32_t min_num_anchors;        /* --min-num-anchors          10   */
  int32_t min_num_anchors_output; /* --min-num-anchors-output   10   */
  float stop_mapping;             /* --stop-mapping             1.4  */
  float stop_mapping_output;      /* --stop-mapping-output      1.2  */
  float stop_mapping_mean;        /* --stop-mapping-mean        5    */
  float stop_mapping_mean_output; /* --stop-mapping-mean-output 5    */
} smb_params;

/* One PAF row's numeric content = `PAFMapping` (output_tools.h:16-38) plus the tag values
 * StreamingMap appends (sigmap.cc:731-745).  Fixed-size, caller-allocated. */
typedef struct smb_mapping {
  uint32_t mapped;      /* 1: mapped row; 0: unmapped row (mapq 61, sigmap.cc:864) */
  uint32_t read_len;    /* kept samples after the (30,200) pA filter: col 2, col 10, sl */
  uint32_t q_start, q_end; /* col 3, 4 */
  uint32_t strand_plus; /* 1 '+', 0 '-' */
  uint32_t contig;      /* reference sequence index */
  uint32_t t_start;     /* col 8 */
  uint32_t frag_len;    /* col 11; col 9 = t_start + frag_len */
  uint32_t mapq;        /* col 12 */
  uint32_t chunks;      /* ci */
  uint32_t n_chains;    /* nc (0 => the row carries only mt/ci/sl) */
  uint32_t cm;          /* anchors in the best chain */
  float s1, s2, sm, ad, at, aq;
  uint32_t num_events;  /* kept events consumed over all chunks */
  uint32_t flags;       /* bit0: some query exceeded SMB_MAX_HITS (H4: order differs) */
} smb_mapping;

/* One chain = `SignalAnchorChain` without the anchor vector (spatial_index.h:28-45). */
typedef struct smb_chain {
  float score;
  uint32_t contig, start, end, n_anchors, mapq;
  uint32_t dir; /* 1 Positive, 0 Negative */
} smb_chain;

/* `SignalAnchor` (spatial_index.h:18-26) */
typedef struct smb_anchor {
  uint32_t target, query;
  float dist;
} smb_anchor;

/* Work counters and device timings of the calls made since smb_stats_reset(). */
typedef struct smb_stats {
  uint64_t samples;        /* S: raw samples consumed in chunks (ci * 4000 summed) */
  uint64_t raw_events;
  uint64_t events;         /* E: kept events */
  uint64_t queries;        /* Q */
  uint64_t hits;           /* H: anchors emitted by the radius search */
  uint64_t anchors;        /* A: anchors entering the DP (H + carried) */
  uint64_t capped_queries; /* queries that hit the 5000 cap */
  uint64_t chunks;         /* chunk invocations */
  uint64_t steps;          /* batched pipeline steps */
  uint64_t launches;       /* CUDA kernels launched by this library */
  double ms_events, ms_search, ms_sort, ms_chain, ms_filter, ms_total; /* CUDA-event ms */
  uint64_t search_launches; /* launches of the radius-search kernel (ms_search / this) */
  uint64_t h2d_bytes, d2h_bytes;
  uint64_t linked;         /* anchors the chaining DP had to walk sequentially (have a
                              gap-compatible predecessor); the rest are settled in parallel */
  uint64_t seg_sort_steps; /* steps whose anchors were sorted per entry in shared memory
                              (the others fell back to the global radix sort) */
  uint64_t exchanges;      /* collectives issued by a contig-sharded run (0 otherwise) */
  uint64_t part_sort_steps; /* of seg_sort_steps: sorted one CTA per (entry, part) from pre-routed runs */
  uint64_t overflow_queries; /* queries whose frontier outgrew the lean search kernel's slots and went
                                through the general one (every query does with option search=general) */
  uint64_t sync_points;     /* host waits on the device inside the mapping calls */
  double ms_stream_stage;   /* host milliseconds smb_stream_round spent filtering / cutting / staging chunks */
  uint64_t pending;         /* of `linked`, the anchors left to the DP kernels (the chain-prep kernel
                               settles the rest itself) */
} smb_stats;

/* ------------------------------------------------------------------ context */
void smb_default_params(smb_params *p);
int smb_device_count(void);             /* CUDA devices visible; 0 without a driver */
int smb_create(smb_ctx **ctx, int device);
void smb_destroy(smb_ctx *ctx);
const char *smb_last_error(const smb_ctx *ctx); /* ctx may be NULL: last create() error */
void smb_stats_reset(smb_ctx *ctx);
int smb_stats_get(smb_ctx *ctx, smb_stats *out);
/* Device-side stopwatch on the library's own stream (CUDA events): start records an event,
 * stop records a second one, synchronises and returns the elapsed milliseconds. */
int smb_timer_start(smb_ctx *ctx);
int smb_timer_stop(smb_ctx *ctx, double *ms);
/* tuning: max chunks per pipeline step and anchor capacity per step (0 = keep default) */
int smb_set_limits(smb_ctx *ctx, uint32_t max_batch_chunks, uint64_t max_batch_anchors);

/* Run-time switches for A/B measurements and for tests that have to reach the fallback paths:
 * name = an SMB_<NAME> environment variable without the prefix (smb_create reads those once),
 * e.g. ("sort", "part|entry|global"), ("search", "lean|general"), ("front_cap", "72"),
 * ("runs_cap", "64"), ("dp_passes", "3"), ("events", "auto|thread|warp").  Results never
 * depend on them (every path is held to the same parity tests); only speed does. */
int smb_set_option(smb_ctx *ctx, const char *name, const char *value);

/* -------------------------------------------------------------------- index */
/* Replaces SpatialIndex::Load (spatial_index.cc:132-163).  Reads <prefix>.pt (the point
 * cloud written by SpatialIndex::Save, :105-123) and builds the flat device index from it;
 * <prefix>.si (nanoflann's KD-tree dump) is not needed and not read. */
int smb_index_load(smb_ctx *ctx, const char *prefix);
/* Same, from an in-memory point cloud: pos[i] = Point::position, val[i] = Point::value
 * (sigmap_adaptor.h:7-17). */
int smb_index_set_points(smb_ctx *ctx, const uint64_t *pos, const float *val, size_t n);
/* Reference sequence lengths (SequenceBatch::GetSequenceLengthAt): needed for the '-'
 * strand coordinate flip (sigmap.cc:754-757) and to size the per-contig buckets. */
int smb_index_set_contigs(smb_ctx *ctx, const uint32_t *lengths, uint32_t n_contigs);
uint64_t smb_index_num_points(const smb_ctx *ctx);

/* ------------------------------------------- contig-sharded index (multi-GPU) */
/* For references whose index exceeds one GPU (SURVEY.md 8e mode 2; the reference itself has no
 * such mode -- its SpatialIndex::Load, spatial_index.cc:132-163, needs the whole KD-tree in one
 * address space).  Contigs are partitioned over `world` ranks; every rank is handed every read
 * (smb_map_reads etc. unchanged), searches and chains against its own contigs, and three small
 * collectives per pipeline step (running max per bucket, chain candidates) make every rank
 * return the rows the unsharded run returns, bit for bit.
 *
 * Group setup, one of:
 *   smb_shard_nccl_init    one process per GPU (torchrun): rank 0 calls smb_shard_nccl_unique_id
 *                          and broadcasts the 128 bytes out of band (torch.distributed, MPI, a
 *                          file); the collectives are NCCL over NVLink on the context's stream.
 *   smb_shard_local_group  n contexts inside one process, each then driven by its own host
 *                          thread; rendezvous on a host barrier + peer copies.
 * Then every rank calls smb_index_set_points_sharded with the SAME full point cloud and owner
 * table (smbh_assign_contigs gives a balanced one) and smb_index_set_contigs as usual; all
 * mapping calls must then be made by every rank with identical arguments. */
int smbh_assign_contigs(const uint32_t *lengths, uint32_t n_contigs, uint32_t world,
                        uint32_t *owner /* n_contigs */);
int smb_shard_local_group(smb_ctx *const *ctxs, uint32_t n);
int smb_shard_nccl_unique_id(char *id128);
int smb_shard_nccl_init(smb_ctx *ctx, int rank, int world, const char *id128);
int smb_shard_rank(const smb_ctx *ctx);
int smb_shard_world(const smb_ctx *ctx);
int smb_index_set_points_sharded(smb_ctx *ctx, const uint64_t *pos, const float *val, size_t n,
                                 const uint32_t *contig_owner, uint32_t n_contigs);
/* The same from the rank's own part of the cloud (smbh_build_point_cloud_part with this context's
 * shard rank): no rank ever needs the whole cloud in host memory. */
struct smbh_cloud_part;
int smb_index_set_points_part(smb_ctx *ctx, const struct smbh_cloud_part *part, uint32_t n_contigs);
uint32_t smb_index_num_contigs(const smb_ctx *ctx);
/* Read-sharded runs (reads split over the GPUs, index replicated; the taskloop of sigmap.cc:618-632
 * spread over devices): the index is built once, on `root`, and copied to the other ranks of the
 * group over NVLink (ncclBroadcast / peer copies) instead of being rebuilt by every rank.  Collective:
 * every member of the group (smb_shard_nccl_init / smb_shard_local_group) calls it; only the root needs
 * smb_index_load / smb_index_set_points + smb_index_set_contigs beforehand.  The mapping calls that
 * follow are independent per rank (no collective on the data path). */
int smb_index_broadcast(smb_ctx *ctx, int root);

/* ------------------------------------------------------- device index build */
/* Sigmap::ConstructIndex (sigmap.cc:999-1046) on this context's GPU: the point cloud of
 * smbh_build_point_cloud_alloc, bit for bit (same pos, val, order), built from the sequences
 * without a host pass.  seqs[i] holds lengths[i] bases followed by a NUL.  *pos / *val are
 * allocated by the library (release with smbh_free). */
int smb_point_cloud_build(smb_ctx *ctx, const char *const *seqs, const uint32_t *lengths, uint32_t n,
                          const float *level_mean, uint64_t **pos, float **val, size_t *count);
/* One rank's part of that cloud, field for field what smbh_build_point_cloud_part fills (free
 * with smbh_cloud_part_free).  Needs no shard group. */
int smb_point_cloud_build_part(smb_ctx *ctx, const char *const *seqs, const uint32_t *lengths, uint32_t n,
                               const float *level_mean, const uint32_t *owner, uint32_t rank,
                               struct smbh_cloud_part *out);
/* The device index straight from the sequences; no point cloud passes through host memory.
 * contig_owner == NULL: the whole index, as smb_index_set_points builds it from the same cloud.
 * Otherwise this context's shard of a contig-sharded index, as smb_index_set_points_sharded builds
 * it (join a shard group first); the device keeps only the rank's part.  Set the contig lengths
 * with smb_index_set_contigs as usual.  SMB_ERR_CAPACITY when the device memory does not hold the
 * build (about 6 bytes per base of the reference and 12 per point of the whole cloud, then the
 * index itself). */
int smb_index_build(smb_ctx *ctx, const char *const *seqs, const uint32_t *lengths, uint32_t n,
                    const float *level_mean, const uint32_t *contig_owner);
/* The last device cloud build of this context.  The `last kept value` selection walks tiles of
 * `tile` window starts (option "cloud_tile") speculatively, then re-walks the tiles whose incoming
 * state it guessed wrong (DESIGN.md, device index build). */
typedef struct smb_build_stats {
  uint64_t points;             /* points of the whole cloud */
  uint64_t tiles;              /* selection tiles */
  uint64_t tiles_rewalked;     /* tiles whose first decisions differed from the speculative walk */
  uint64_t tiles_unconverged;  /* tiles that passed their incoming state on (all masked, or never
                                  met the speculative walk: a run of equal z) */
  uint64_t tiles_redone;       /* tiles re-walked a second time, behind an unconverged one */
  uint64_t tile;               /* window starts per tile */
  uint32_t strands;            /* strands with a window (2 per contig of >= 11 bases) */
  uint32_t strands_serial_mean; /* of those, strands whose level sum could not be taken as an exact
                                   integer sum and was added sequentially (DESIGN.md) */
  double ms_upload, ms_census, ms_levels, ms_zsums, ms_select, ms_scatter, ms_index; /* CUDA-event ms */
} smb_build_stats;
int smb_index_build_stats(smb_ctx *ctx, smb_build_stats *out);

/* ------------------------------------------------------------ whole hot path */
/* Replaces the per-read body of Sigmap::StreamingMap (sigmap.cc:630-866) for n_reads
 * reads at once: raw int16 samples of read r are raw[read_off[r] .. read_off[r+1]);
 * digitisation/range/offset are the per-read SLOW5 fields (signal_batch.cc:187-191).
 * raw is a host pointer (copied in, pinned or pageable); samples already in device memory go
 * through smb_map_reads_device.  out[r] receives read r's row. */
int smb_map_reads(smb_ctx *ctx, const int16_t *raw, const uint64_t *read_off,
                  const float *digitisation, const float *range, const float *offset,
                  size_t n_reads, const smb_params *params, smb_mapping *out);
/* smb_map_reads for samples already in device memory on this context's device.  Read r is
 * raw[read_start[r] .. read_start[r] + read_len[r]) (int16 elements; reads may be in any order,
 * have gaps between them, or be the rows of a padded [n_reads][stride] tensor).  read_start,
 * read_len, digitisation, range, offset and out are host arrays.  The library reads raw and
 * never writes it; the samples are not copied.  stream (a cudaStream_t, may be NULL for the legacy
 * default stream): the call's device work is ordered after what is queued on it.  raw may be
 * reused by the caller when the call returns.  Rows are those smb_map_reads returns for the same
 * samples, bit for bit.
 * raw must be device (or managed) memory of the context's device, else SMB_ERR_ARG; it is neither
 * read nor checked when every read_len is 0 (such a read gets an unmapped row).  Precondition the
 * library cannot check: every read lies inside the caller's allocation.
 * Afterwards the context holds no uploaded read set: smb_map_uploaded returns SMB_ERR_STATE until
 * the next smb_reads_upload or smb_map_reads. */
int smb_map_reads_device(smb_ctx *ctx, const int16_t *raw, const uint64_t *read_start,
                         const uint32_t *read_len, const float *digitisation, const float *range,
                         const float *offset, size_t n_reads, const smb_params *params,
                         smb_mapping *out, void *stream);
/* Two-phase variant used to time with inputs resident in HBM: upload once, map many. */
int smb_reads_upload(smb_ctx *ctx, const int16_t *raw, const uint64_t *read_off,
                     const float *digitisation, const float *range, const float *offset,
                     size_t n_reads);
int smb_map_uploaded(smb_ctx *ctx, const smb_params *params, smb_mapping *out);

/* ------------------------------------------------------------- stage hooks */
/* K1 = SignalBatch::AddSignal (signal_batch.cc:182-210): pA conversion, (30,200) filter,
 * compaction.  out must hold n floats; *n_out = kept samples. */
int smb_stage_raw_to_pa(smb_ctx *ctx, const int16_t *raw, size_t n, float digitisation,
                        float offset, float range, float *out, size_t *n_out);
/* K2/K3 = Sigmap::GenerateEvents (sigmap.cc:1048-1083) on n_chunks chunks of SMB_CHUNK
 * pA samples each (chunk-major).  features: n_chunks x SMB_CHUNK floats (row c holds
 * n_features[c] values). */
int smb_stage_events(smb_ctx *ctx, const float *pa, size_t n_chunks, float *features,
                     uint32_t *n_features);
/* Debug view of event.h:226 DetectEvents for ONE chunk: t-statistics (SMB_CHUNK+1 each),
 * peak positions, raw event means.  Any output pointer may be NULL. */
int smb_stage_detect(smb_ctx *ctx, const float *pa, float *tstat1, float *tstat2,
                     uint32_t *peaks, uint32_t *n_peaks, float *means, uint32_t *n_events);
/* K4 = index->radiusSearch(q, radius, out, sorted=false) (spatial_index.cc:366) for nq
 * queries of SMB_DIM floats.  Hits of query k are hit_idx/hit_d2[hit_off[k]..hit_off[k+1]),
 * sorted by point index (the reference's KD traversal order is not reproducible; compare
 * as sets).  No 5000 cap is applied here.  cap = capacity of hit_idx/hit_d2. */
int smb_stage_radius(smb_ctx *ctx, const float *queries, size_t nq, float radius,
                     uint64_t *hit_off, uint64_t *hit_idx, float *hit_d2, uint64_t cap);

/* K4..K7 = SpatialIndex::GenerateChains (spatial_index.cc:276-577) with the `chains`
 * in/out argument held on the device per read slot.  A batch owns n_slots slots. */
int smb_batch_create(smb_ctx *ctx, uint32_t n_slots, smb_batch **batch);
void smb_batch_destroy(smb_batch *batch);
int smb_batch_reset(smb_batch *batch); /* chains.clear(), num_events = 0 on every slot */
/* For each i < n: GenerateChains(features[feat_off[i]..feat_off[i+1]), num_events[slot],
 * step, radius, n_contigs, chains[slot]) and num_events[slot] += n_features, exactly as
 * sigmap.cc:660-666 (entries with <= 50 features are skipped like the reference does). */
int smb_batch_generate_chains(smb_batch *batch, const uint32_t *slots, uint32_t n,
                              const float *features, const uint32_t *feat_off,
                              const smb_params *params);
int smb_batch_chain_count(smb_batch *batch, uint32_t slot, uint32_t *n_chains);
int smb_batch_get_chains(smb_batch *batch, uint32_t slot, smb_chain *out, uint32_t cap);
int smb_batch_get_anchors(smb_batch *batch, uint32_t slot, uint32_t chain, smb_anchor *out,
                          uint32_t cap);

/* ---------------------------------------------------------------- streaming */
/* Read-until style rounds (sigmap.cc:647-688 turned inside out): every call feeds raw
 * samples of some channels; a channel maps each completed 4000-kept-sample chunk and
 * reports the stop decision.  decisions[i]: 0 keep sequencing, 1 stop (mapped decision
 * reached), per input entry; maps[i] is the row the read would get if it ended now. */
int smb_stream_open(smb_ctx *ctx, uint32_t n_channels, const smb_params *params);
int smb_stream_begin_read(smb_ctx *ctx, uint32_t channel, float digitisation, float range,
                          float offset);
int smb_stream_round(smb_ctx *ctx, const uint32_t *channels, uint32_t n,
                     const int16_t *samples, const uint32_t *sample_off,
                     uint8_t *decisions, smb_mapping *maps);
int smb_stream_close(smb_ctx *ctx);

/* ============================ host-only helpers (no GPU) ==================== */
/* PAF text of one row: PAFOutputTools<PAFMapping>::AppendMapping / AppendUnmappedRead
 * (output_tools.h:200-210,336-354) + tags (sigmap.cc:731-745).  Returns bytes written. */
int smbh_format_paf(const smb_mapping *m, const char *read_name, const char *contig_name,
                    uint32_t contig_len, double mt_ms, char *buf, size_t cap);
/* Pore model TSV (pore_model.cc:11-47): fills 4096 level means / stdvs by 2-bit 6-mer hash */
int smbh_pore_model_load(const char *path, float *level_mean, float *level_stdv);
/* FASTA (plain or gz) -> names/lengths/sequences; free with smbh_fasta_free */
typedef struct smbh_fasta {
  uint32_t n;
  char **names;
  char **seqs;
  uint32_t *lengths;
} smbh_fasta;
int smbh_fasta_load(const char *path, smbh_fasta *out);
void smbh_fasta_free(smbh_fasta *f);
int smbh_fasta_write(const char *path, const char *const *names, const char *const *seqs,
                     const uint32_t *lengths, uint32_t n);
/* Point cloud of Sigmap::ConstructIndex (sigmap.cc:999-1046, spatial_index.cc:33-93).
 * Call with pos == NULL to get the count. */
size_t smbh_build_point_cloud(const char *const *seqs, const uint32_t *lengths, uint32_t n,
                              const float *level_mean, uint64_t *pos, float *val);
/* The same in one pass: *pos / *val are allocated by the library (release with smbh_free). */
int smbh_build_point_cloud_alloc(const char *const *seqs, const uint32_t *lengths, uint32_t n,
                                 const float *level_mean, uint64_t **pos, float **val, size_t *count);
/* One rank's part of the point cloud for a contig-sharded index: the points of the contigs with
 * owner[c] == rank and, after each stretch of them, the SMB_DIM-1 points that follow in the whole
 * cloud (the last windows of the stretch straddle into them, Q2), as runs of consecutive cloud points.
 * Run k = values [run_off[k], run_off[k+1]), its first point is point run_first[k] of the whole cloud;
 * own[i] = 1 where point i belongs to the rank (only those start windows).  A rank of a genome-scale
 * job holds its share of the cloud, never the whole (3.1 Gbp: 74 GB).  Free with smbh_cloud_part_free. */
typedef struct smbh_cloud_part {
  size_t n_values, n_runs;
  uint64_t n_points_total; /* size of the whole cloud */
  uint64_t *pos;
  float *val;
  uint8_t *own;
  uint64_t *run_off;   /* n_runs + 1 */
  uint64_t *run_first; /* n_runs */
} smbh_cloud_part;
int smbh_build_point_cloud_part(const char *const *seqs, const uint32_t *lengths, uint32_t n,
                                const float *level_mean, const uint32_t *owner, uint32_t rank,
                                smbh_cloud_part *out);
void smbh_cloud_part_free(smbh_cloud_part *p);
/* .pt file of SpatialIndex::Save (spatial_index.cc:105-123) */
int smbh_pt_write(const char *prefix, const uint64_t *pos, const float *val, size_t n,
                  int dim, int max_leaf);
int smbh_pt_read(const char *prefix, uint64_t **pos, float **val, size_t *n, int *dim,
                 int *max_leaf);
/* <prefix>.si: a KD-tree over the window points in the layout of nanoflann's saveIndex_
 * (nanoflann.hpp:1051-1058), so that the reference's own `sigmap -m` (SpatialIndex::Load,
 * spatial_index.cc:132-163) can load an index written by this program.  This library never reads it. */
int smbh_si_write(const char *prefix, const float *val, size_t n_points, int dim, int max_leaf);
void smbh_free(void *p);
/* BLOW5 (slow5lib 0.2.0 binary layout, uncompressed or zlib records) */
typedef struct smbh_reads {
  size_t n;
  char **names;
  uint64_t *read_off; /* n+1 */
  int16_t *raw;
  float *digitisation, *range, *offset;
} smbh_reads;
int smbh_blow5_write(const char *path, const char *const *names, const int16_t *raw,
                     const uint64_t *read_off, size_t n, double digitisation, double offset,
                     double range, double sampling_rate);
int smbh_blow5_read(const char *path, smbh_reads *out); /* appends to *out (zero-init first) */
/* message of the last failed smbh_* call on this thread (BLOW5 version / compression, ...) */
const char *smbh_last_error(void);
void smbh_reads_free(smbh_reads *r);
/* Synthetic data (SURVEY.md 8d): uniform ACGT reference, reads simulated from the
 * 6-mer model.  Deterministic in (seed, read index) so ranks can generate disjoint read
 * ranges.  sim_reads: first call with raw == NULL fills read_off (n+1) only. */
int smbh_sim_reference(uint64_t seed, const uint32_t *lengths, uint32_t n_contigs,
                       char **seqs /* caller-allocated, lengths[i]+1 bytes each */);
int smbh_sim_reads(uint64_t seed, const char *const *seqs, const uint32_t *lengths,
                   uint32_t n_contigs, const float *level_mean, const float *level_stdv,
                   uint64_t first_read, uint64_t n_reads, uint32_t min_bases,
                   uint32_t max_bases, float noise, uint64_t *read_off, int16_t *raw,
                   uint32_t *truth /* n_reads x 4: contig,start,end,strand_plus; may be NULL */);

#ifdef __cplusplus
}
#endif
#endif /* SIGMAP_B200_H */
