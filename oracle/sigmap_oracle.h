/*
 * oracle/sigmap_oracle.h -- CPU restatement of the reference's per-read mapping
 * hot path.  TEST INFRASTRUCTURE ONLY: tests/, __graft_entry__.smoke() and the
 * cpu_baseline leg of bench.py may load it; the product (sigmap_b200/) never does.
 *
 * Parity pin: this restatement is checked bit-for-bit against the UNMODIFIED
 * reference compiled by oracle/Makefile (oracle/_ref/libsigmap_ref_stage.so and
 * oracle/_ref/sigmap_ref, strict-FP build) by tests/make_golden.py, and the
 * resulting vectors are committed under tests/golden/.  The reference ships no
 * golden vectors of its own for this path (SURVEY.md 8c).
 */
#ifndef SIGMAP_ORACLE_H
#define SIGMAP_ORACLE_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct {
  uint32_t target, query;
  float dist;
} orc_anchor;

typedef struct {
  float score;
  uint32_t contig, start, end, n_anchors;
  uint32_t mapq;
  uint32_t dir; /* 1 = Positive (+), 0 = Negative (-): spatial_index.h:13-16 */
  orc_anchor *anchors; /* end -> start order, n_anchors entries (malloc'ed) */
} orc_chain;

typedef struct {
  orc_chain *chains;
  size_t n, cap;
} orc_chain_list;

/* StreamingMap knobs: sigmap.cc:1380-1419 defaults */
typedef struct {
  float search_radius;          /* 0.08 */
  int step;                     /* 2 */
  int max_num_chunks;           /* 30 */
  int stop_min_anchors;         /* 10 */
  int output_min_anchors;       /* 10 */
  float stop_ratio;             /* 1.4 */
  float output_ratio;           /* 1.2 */
  float stop_mean_ratio;        /* 5 */
  float output_mean_ratio;      /* 5 */
} orc_params;

typedef struct {
  int mapped;                 /* 1 -> mapped PAF row, 0 -> unmapped row (mapq 61) */
  uint32_t read_len;          /* kept (filtered) samples: PAF col 2 and tag sl */
  uint32_t q_start, q_end;    /* PAF col 3,4 */
  uint32_t strand_plus;       /* 1 '+', 0 '-' */
  uint32_t contig;
  uint32_t t_start, frag_len; /* PAF col 8; col 9 = t_start+frag_len; col 11 = frag_len */
  uint32_t mapq;
  uint32_t chunks;            /* tag ci */
  uint32_t n_chains;          /* tag nc (0 -> no chain tags on unmapped rows) */
  uint32_t cm;                /* anchors in best chain */
  float s1, s2, sm, ad, at, aq;
  uint32_t num_events;        /* kept events consumed (query offset at the end) */
} orc_mapping;

/* What the chaining of spatial_index.cc:411-576 met, for tests that must show their data
 * reaches the rare branches of the CUDA chaining.  Filled by the *_counted entry points when
 * given a non-NULL pointer: counts add up over calls, the maxima keep the largest value. */
typedef struct {
  uint64_t max_query_hits;     /* most hits one query found (the reference keeps 5 000: :371-372) */
  uint64_t max_bucket_anchors; /* largest (contig, strand) bucket of a chunk, carried anchors included */
  /* the lookback of :434-540 */
  uint64_t walks_band;         /* lookbacks that ran to start = i - band > 0 */
  uint64_t walks_skips;        /* lookbacks ended by skips > max_skips */
  uint64_t walks_target_gap;   /* lookbacks ended by a target gap > 5 000 */
  uint64_t longest_walk;       /* most predecessors one lookback visited */
  /* anchors whose position-only lookback range (same bucket, band, target gap, and
   * 3 dt < 4 (q_i - qmin) with qmin the chunk's query offset lowered by the bucket's carried
   * anchors) holds more than 1 152 predecessors and no gap-compatible one */
  uint64_t deep_link_ranges;
  uint64_t traceback_hit_used; /* chains emitted with score[end] - score[pred] (:165-220) */
  uint64_t end_ties;           /* top-3 end picks decided by index between equal scores (:552-568) */
  uint64_t primary_ties;       /* adjacent equal scores after the primary sort (:222-253) */
} orc_chain_counters;

void orc_default_params(orc_params *p);

/* A.0  signal_batch.cc:182-210 */
size_t orc_raw_to_pa(const int16_t *raw, size_t n, double digitisation, double offset,
                     double range, float *out);
/* A.1  event.h:58-267 ; returns number of raw events.  tstat arrays have n+1 entries. */
size_t orc_detect_events(const float *x, size_t n, float *tstat1, float *tstat2,
                         uint64_t *peaks, size_t *n_peaks, float *means, uint64_t *starts,
                         uint64_t *lengths);
/* A.1  sigmap.cc:1048-1083,1131-1155 ; returns number of kept (compressed) features */
size_t orc_generate_events(const float *x, size_t n, float *features);
/* A.2  nanoflann.hpp:383-408,249-251 by brute force over the N-5 windows, index order */
size_t orc_radius_search(const float *vals, size_t n_points, const float *q, float radius,
                         uint64_t *idx_out, float *d2_out, size_t cap);
/* A.2+A.3  spatial_index.cc:276-577 ; `chains` is in/out like the reference's argument */
void orc_generate_chains(const uint64_t *pos, const float *vals, size_t n_points,
                         const float *features, size_t n_features, uint32_t query_offset,
                         int step, float radius, size_t n_targets, orc_chain_list *chains);
void orc_generate_chains_counted(const uint64_t *pos, const float *vals, size_t n_points,
                                 const float *features, size_t n_features, uint32_t query_offset,
                                 int step, float radius, size_t n_targets, orc_chain_list *chains,
                                 orc_chain_counters *ctr);
/* same but with the hit lists supplied by the caller (per query: first hit index into
 * hit_idx/hit_d2 = hit_off[k], count = hit_off[k+1]-hit_off[k]); lets tests drive A.3
 * with the reference's own KD-tree hit order */
void orc_chain_from_hits(const uint64_t *pos, const uint32_t *query_pos, size_t n_queries,
                         const uint64_t *hit_off, const uint64_t *hit_idx, const float *hit_d2,
                         float radius, size_t n_targets, orc_chain_list *chains);
void orc_chain_list_free(orc_chain_list *l);
/* A.4  sigmap.cc:637-865 for one read given its kept pA samples */
void orc_streaming_map(const uint64_t *pos, const float *vals, size_t n_points,
                       size_t n_targets, const uint32_t *contig_len, const float *pa,
                       size_t n_pa, const orc_params *p, orc_mapping *out);
void orc_streaming_map_counted(const uint64_t *pos, const float *vals, size_t n_points,
                               size_t n_targets, const uint32_t *contig_len, const float *pa,
                               size_t n_pa, const orc_params *p, orc_mapping *out,
                               orc_chain_counters *ctr);
/* A.4  output_tools.h:200-210,336-354 + sigmap.cc:731-745 ; mt tag printed as given */
int orc_format_paf(const orc_mapping *m, const char *read_name, const char *contig_name,
                   uint32_t contig_len, double mt_ms, char *buf, size_t cap);
/* A.5  pore_model.cc:57-80 (Q1), sigmap.cc:19-185,1131-1155, spatial_index.cc:33-93.
 * seqs: n_seq NUL-terminated sequences.  level_mean: 4096 fp32 6-mer means indexed by the
 * 2-bit hash (A=0,C=1,G=2,T=3).  Returns number of points written (call with pos==NULL to
 * count). */
size_t orc_build_point_cloud(const char *const *seqs, const uint32_t *seq_len, size_t n_seq,
                             const float *level_mean, uint64_t *pos, float *vals);

#ifdef __cplusplus
}
#endif
#endif
