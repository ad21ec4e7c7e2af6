/*
 * oracle/sigmap_oracle.c -- plain-C CPU restatement of Sigmap's per-read mapping hot
 * path (raw signal -> events -> radius search -> anchors -> chaining -> decision).
 *
 * TEST INFRASTRUCTURE ONLY.  Loaded by tests/, __graft_entry__.smoke() and the
 * cpu_baseline leg of bench.py as the checker; never by the product.
 *
 * Parity pin: every function below is checked bit-for-bit by tests/make_golden.py
 * against the unmodified reference objects (oracle/_ref/, strict-FP build
 * `-O3 -ffp-contract=off`, no -march=native).  The reference repository holds no
 * golden vectors for this path; the vectors under tests/golden/ were produced by the
 * reference itself in the build container.
 *
 * Must be compiled with -ffp-contract=off on a target whose float arithmetic is IEEE
 * binary32 (x86-64 SSE): the last-ulp behaviour of the fp32 prefix sums and of the
 * double-precision sqrt/fabs in the t-statistic decides parity (SURVEY.md H1, Q6).
 */
#include "sigmap_oracle.h"

#include <float.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define DIM 6

void orc_default_params(orc_params *p) { /* sigmap.cc:1380-1419 */
  p->search_radius = 0.08f;
  p->step = 2;
  p->max_num_chunks = 30;
  p->stop_min_anchors = 10;
  p->output_min_anchors = 10;
  p->stop_ratio = 1.4f;
  p->output_ratio = 1.2f;
  p->stop_mean_ratio = 5;
  p->output_mean_ratio = 5;
}

/* ------------------------------------------------------------------ A.0 */
/* signal_batch.cc:182-210: float offset/scale, keep iff 30 < pA < 200 */
size_t orc_raw_to_pa(const int16_t *raw, size_t n, double digitisation, double offset_d,
                     double range_d, float *out) {
  float dig = (float)digitisation, range = (float)range_d, offset = (float)offset_d;
  float scale = range / dig;
  size_t k = 0;
  for (size_t i = 0; i < n; ++i) {
    float pa = ((float)raw[i] + offset) * scale;
    if (pa > 30 && pa < 200) out[k++] = pa;
  }
  return k;
}

/* ------------------------------------------------------------------ A.1 */
/* event.h:58-68 */
static void prefix_sums(const float *x, size_t n, float *ps, float *pss) {
  ps[0] = 0.0f;
  pss[0] = 0.0f;
  for (size_t i = 0; i < n; ++i) {
    ps[i + 1] = ps[i] + x[i];
    float sq = x[i] * x[i];
    pss[i + 1] = pss[i] + sq;
  }
}

/* event.h:70-115; returns the number of entries written (n+1, or n on the quick return) */
static size_t tstat(const float *ps, const float *pss, size_t n, size_t w, float *t) {
  const float eta = FLT_MIN;
  size_t k = 0;
  if (n < 2 * w || w < 2) {
    for (size_t i = 0; i < n; ++i) t[k++] = 0.0f;
    return k;
  }
  for (size_t i = 0; i < w; ++i) t[k++] = 0.0f;
  const float wf = (float)w;
  for (size_t i = w; i <= n - w; ++i) {
    float sum1 = ps[i], sumsq1 = pss[i];
    if (i > w) {
      sum1 -= ps[i - w];
      sumsq1 -= pss[i - w];
    }
    float sum2 = ps[i + w] - ps[i];
    float sumsq2 = pss[i + w] - pss[i];
    float mean1 = sum1 / wf, mean2 = sum2 / wf;
    float a = sumsq1 / wf, b = mean1 * mean1, c = sumsq2 / wf, d = mean2 * mean2;
    float cv = ((a - b) + c) - d; /* event.h:100-101 association */
    cv = fmaxf(cv, eta);
    float dm = mean2 - mean1;
    float cvw = cv / wf;
    /* Q6: fabs/sqrt resolve to the double versions in the shipped TU */
    t[k++] = (float)(fabs((double)dm) / sqrt((double)cvw));
  }
  for (size_t i = 0; i < w; ++i) t[k++] = 0.0f;
  return k;
}

typedef struct {
  const float *sig;
  float thr;
  size_t w, masked_to;
  int peak_pos;
  float peak_value;
  int valid;
} detector;

/* event.h:117-182 */
static size_t find_peaks(const float *t1, const float *t2, size_t n, uint64_t *peaks) {
  detector d[2] = {{t1, 4.30265f, 3, 0, -1, FLT_MAX, 0}, {t2, 2.57058f, 6, 0, -1, FLT_MAX, 0}};
  const float peak_height = 1.0f;
  size_t np = 0;
  for (size_t i = 0; i < n; ++i) {
    for (int k = 0; k < 2; ++k) {
      detector *x = &d[k];
      if (x->masked_to >= i) continue;
      float cur = x->sig[i];
      if (x->peak_pos == -1) {
        if (cur < x->peak_value) {
          x->peak_value = cur;
        } else if (cur - x->peak_value > peak_height) {
          x->peak_value = cur;
          x->peak_pos = (int)i;
        }
      } else {
        if (cur > x->peak_value) {
          x->peak_value = cur;
          x->peak_pos = (int)i;
        }
        if (k == 0 && x->peak_value > x->thr) {
          d[1].masked_to = (size_t)x->peak_pos + x->w;
          d[1].peak_pos = -1;
          d[1].peak_value = FLT_MAX;
          d[1].valid = 0;
        }
        if (x->peak_value - cur > peak_height && x->peak_value > x->thr) x->valid = 1;
        if (x->valid && (i - (size_t)x->peak_pos) > x->w / 2) {
          peaks[np++] = (uint64_t)x->peak_pos;
          x->peak_pos = -1;
          x->peak_value = cur;
          x->valid = 0;
        }
      }
    }
  }
  return np;
}

/* event.h:184-198 (stdv is computed by the reference but never read downstream: Q7) */
static float event_mean(uint64_t s, uint64_t e, const float *ps) {
  uint64_t len = e - s; /* unsigned wrap kept as in the reference */
  return (ps[e] - ps[s]) / (float)len;
}

size_t orc_detect_events(const float *x, size_t n, float *tstat1, float *tstat2,
                         uint64_t *peaks, size_t *n_peaks, float *means, uint64_t *starts,
                         uint64_t *lengths) {
  float *ps = (float *)malloc((n + 1) * sizeof(float));
  float *pss = (float *)malloc((n + 1) * sizeof(float));
  float *t1 = tstat1 ? tstat1 : (float *)malloc((n + 1) * sizeof(float));
  float *t2 = tstat2 ? tstat2 : (float *)malloc((n + 1) * sizeof(float));
  uint64_t *pk = peaks ? peaks : (uint64_t *)malloc((2 * n + 2) * sizeof(uint64_t));
  prefix_sums(x, n, ps, pss);
  tstat(ps, pss, n, 3, t1);
  tstat(ps, pss, n, 6, t2);
  size_t np = find_peaks(t1, t2, n, pk);
  if (n_peaks) *n_peaks = np;
  size_t ne = 0;
  /* event.h:200-224.  The reference reads peaks[0] and peaks[num_events-2]
   * unconditionally (undefined behaviour below two peaks); the restatement returns
   * no events there, which StreamingMap treats like any chunk with <= 50 features. */
  if (np >= 2) {
    size_t cnt = 1;
    for (size_t i = 1; i < np; ++i)
      if (pk[i] > 0 && pk[i] < n) cnt++;
    ne = cnt;
    for (size_t k = 0; k < ne; ++k) {
      uint64_t s = (k == 0) ? 0 : pk[k - 1];
      uint64_t e = (k == ne - 1) ? n : pk[k];
      if (means) means[k] = event_mean(s, e, ps);
      if (starts) starts[k] = s;
      if (lengths) lengths[k] = e - s;
    }
  }
  free(ps);
  free(pss);
  if (!tstat1) free(t1);
  if (!tstat2) free(t2);
  if (!peaks) free(pk);
  return ne;
}

/* sigmap.cc:1131-1155 */
static void zscore(const float *x, size_t n, float *out) {
  double mean = 0;
  for (size_t i = 0; i < n; ++i) mean += x[i];
  mean /= n;
  double sd = 0;
  for (size_t i = 0; i < n; ++i) sd += (x[i] - mean) * (x[i] - mean);
  sd /= (n - 1);
  sd = sqrt(sd);
  for (size_t i = 0; i < n; ++i) out[i] = (float)((x[i] - mean) / sd);
}

/* sigmap.cc:1048-1083 */
size_t orc_generate_events(const float *x, size_t n, float *features) {
  float *means = (float *)malloc((n + 2) * sizeof(float));
  size_t ne = orc_detect_events(x, n, NULL, NULL, NULL, NULL, means, NULL, NULL);
  if (ne == 0) {
    free(means);
    return 0;
  }
  float *z = (float *)malloc(ne * sizeof(float));
  zscore(means, ne, z);
  size_t k = 0;
  for (size_t i = 0; i < ne; ++i) {
    /* Q5: float abs, then compared with the double literal 0.1 */
    if (i == 0 || (double)fabsf(z[i] - features[k - 1]) > 0.1) features[k++] = z[i];
  }
  free(means);
  free(z);
  return k;
}

/* ------------------------------------------------------------------ A.2 */
/* nanoflann.hpp:383-408: ((e0+e1)+e2)+e3, then +e4, +e5, all fp32 */
static inline float dist2(const float *q, const float *v) {
  float d0 = q[0] - v[0], d1 = q[1] - v[1], d2 = q[2] - v[2], d3 = q[3] - v[3];
  float e0 = d0 * d0, e1 = d1 * d1, e2 = d2 * d2, e3 = d3 * d3;
  float r = ((e0 + e1) + e2) + e3;
  float d4 = q[4] - v[4];
  float e4 = d4 * d4;
  r = r + e4;
  float d5 = q[5] - v[5];
  float e5 = d5 * d5;
  r = r + e5;
  return r;
}

size_t orc_radius_search(const float *vals, size_t n_points, const float *q, float radius,
                         uint64_t *idx_out, float *d2_out, size_t cap) {
  size_t cnt = 0;
  if (n_points < DIM) return 0;
  for (size_t i = 0; i + DIM <= n_points; ++i) {
    /* exact prefilter: fp32 partial sums are monotone, so e0 >= r already rejects */
    float d0 = q[0] - vals[i];
    if (d0 * d0 >= radius) continue;
    float d = dist2(q, vals + i);
    if (d < radius) { /* nanoflann.hpp:249-251, :1362 strict < */
      if (cnt < cap) {
        idx_out[cnt] = i;
        d2_out[cnt] = d;
      }
      cnt++;
    }
  }
  return cnt;
}

/* ------------------------------------------------------------------ A.3 */
typedef struct {
  orc_anchor *a;
  size_t n, cap;
} bucket;

static void bucket_push(bucket *b, orc_anchor x) {
  if (b->n == b->cap) {
    b->cap = b->cap ? 2 * b->cap : 64;
    b->a = (orc_anchor *)realloc(b->a, b->cap * sizeof(orc_anchor));
  }
  b->a[b->n++] = x;
}

static int anchor_cmp(const void *pa, const void *pb) { /* spatial_index.h:22-25 */
  const orc_anchor *a = (const orc_anchor *)pa, *b = (const orc_anchor *)pb;
  if (a->target != b->target) return a->target < b->target ? -1 : 1;
  if (a->query != b->query) return a->query < b->query ? -1 : 1;
  if (a->dist != b->dist) return a->dist < b->dist ? -1 : 1;
  return 0;
}

static void chains_push(orc_chain_list *l, orc_chain c) {
  if (l->n == l->cap) {
    l->cap = l->cap ? 2 * l->cap : 16;
    l->chains = (orc_chain *)realloc(l->chains, l->cap * sizeof(orc_chain));
  }
  l->chains[l->n++] = c;
}

void orc_chain_list_free(orc_chain_list *l) {
  for (size_t i = 0; i < l->n; ++i) free(l->chains[i].anchors);
  free(l->chains);
  l->chains = NULL;
  l->n = l->cap = 0;
}

/* spatial_index.h:38-44: a > b on (score, n, dir, contig, start, end) */
static int chain_greater(const orc_chain *a, const orc_chain *b) {
  if (a->score != b->score) return a->score > b->score;
  if (a->n_anchors != b->n_anchors) return a->n_anchors > b->n_anchors;
  if (a->dir != b->dir) return a->dir > b->dir;
  if (a->contig != b->contig) return a->contig > b->contig;
  if (a->start != b->start) return a->start > b->start;
  return a->end > b->end;
}

/* spatial_index.cc:165-220 */
static void traceback(uint32_t dir, size_t end_i, uint32_t contig, const float *score,
                      const size_t *pred, const orc_anchor *A, unsigned char *used,
                      orc_chain_list *out, orc_chain_counters *ctr) {
  if (used[end_i]) return;
  size_t cap = 128, n = 0;
  orc_anchor *list = (orc_anchor *)malloc(cap * sizeof(orc_anchor));
  int hit_used = 0;
  size_t s = end_i;
  list[n++] = A[s];
  if (pred[s] != s && used[pred[s]]) hit_used = 1;
  used[s] = 1;
  while (pred[s] != s && !used[pred[s]]) {
    s = pred[s];
    if (n == cap) {
      cap *= 2;
      list = (orc_anchor *)realloc(list, cap * sizeof(orc_anchor));
    }
    list[n++] = A[s];
    if (pred[s] != s && used[pred[s]]) hit_used = 1;
    used[s] = 1;
  }
  if (n >= 2) { /* min_num_anchors = 2, spatial_index.cc:288 */
    float sc = score[end_i];
    if (hit_used) {
      sc -= score[pred[s]];
      if (ctr) ctr->traceback_hit_used++;
    }
    orc_chain c;
    c.score = sc;
    c.contig = contig;
    c.start = A[s].target;
    c.end = A[end_i].target;
    c.n_anchors = (uint32_t)n;
    c.mapq = 0;
    c.dir = dir;
    c.anchors = list;
    chains_push(out, c);
  } else {
    free(list);
  }
}

/* Counters only: the position-only lookback range of anchor i (the range the CUDA chain
 * preparation tests for a gap-compatible predecessor): 1 when it holds more than 1 152
 * predecessors and none of them is gap-compatible. */
static int deep_link_range(const orc_anchor *A, size_t i, int band, int max_target_gap,
                           int max_gap, uint32_t qmin) {
  int32_t ct = (int32_t)A[i].target, cq = (int32_t)A[i].query;
  int64_t qlim = 4 * ((int64_t)cq - (int64_t)qmin);
  size_t depth = i < (size_t)band ? i : (size_t)band, d;
  for (d = 1; d <= depth; ++d) {
    int32_t pt = (int32_t)A[i - d].target, pq = (int32_t)A[i - d].query;
    if (pt + max_target_gap < ct || 3 * (int64_t)(ct - pt) >= qlim) break;
    int32_t dt = ct - pt, dq = cq - pq;
    if (abs(dt - dq) < max_gap && dq < 5 * dt && 4 * dq > 3 * dt) return 0;
  }
  return d - 1 > 1152;
}

/* spatial_index.cc:411-576 given filled buckets [strand][contig]; query_offset is the
 * chunk's first query position (for the counters only) */
static void chain_buckets(bucket *bk[2], size_t n_targets, float radius, uint32_t query_offset,
                          orc_chain_list *chains, orc_chain_counters *ctr) {
  const int max_gap_length = 2000, max_target_gap_length = 5000, band = 5000, max_skips = 25;
  const int num_best = 3;
  const float min_score = 10;
  for (size_t t = 0; t < n_targets; ++t)
    for (int s = 0; s < 2; ++s)
      if (bk[s][t].n > 1) qsort(bk[s][t].a, bk[s][t].n, sizeof(orc_anchor), anchor_cmp);
  float gmax = 0;
  for (size_t t = 0; t < n_targets; ++t) {
    for (int s = 0; s < 2; ++s) {
      const orc_anchor *A = bk[s][t].a;
      size_t n = bk[s][t].n;
      if (n == 0) continue; /* nothing observable happens for an empty bucket */
      uint32_t qmin = query_offset;
      if (ctr) {
        if (n > ctr->max_bucket_anchors) ctr->max_bucket_anchors = n;
        for (size_t i = 0; i < n; ++i)
          if (A[i].query < qmin) qmin = A[i].query;
      }
      float *score = (float *)malloc(n * sizeof(float));
      size_t *pred = (size_t *)malloc(n * sizeof(size_t));
      unsigned char *used = (unsigned char *)calloc(n, 1);
      size_t n_ends = 0, cap_ends = 16;
      float *end_score = (float *)malloc(cap_ends * sizeof(float));
      size_t *end_idx = (size_t *)malloc(cap_ends * sizeof(size_t));
      for (size_t i = 0; i < n; ++i) {
        /* :438-444: double expression rounded to float */
        float coef = (float)(1 - 0.2 * A[i].dist / radius);
        score[i] = coef * (float)DIM;
        pred[i] = i;
        int32_t ct = (int32_t)A[i].target, cq = (int32_t)A[i].query;
        int32_t start = 0;
        if (i > (size_t)band) start = (int32_t)i - band;
        int32_t skips = 0, j;
        int stop = 0; /* counters: 1 target gap, 2 skips */
        for (j = (int32_t)i - 1; j >= start; --j) {
          int32_t pt = (int32_t)A[j].target, pq = (int32_t)A[j].query;
          if (pq == cq) continue;
          if (pt == ct) continue;
          if (pt + max_target_gap_length < ct) {
            stop = 1;
            break;
          }
          int32_t dt = ct - pt, dq = cq - pq;
          float cur = 0;
          if (dq < 0) continue;
          int32_t m = dt < dq ? dt : dq;
          if (m > DIM) m = DIM;
          float matching = (float)m * coef;
          int gap = abs(dt - dq);
          float gap_scale = dt > 0 ? (float)dq / (float)dt : 1;
          if (gap < max_gap_length && gap_scale < 5 && gap_scale > 0.75) cur = score[j] + matching;
          if (cur > score[i]) {
            score[i] = cur;
            pred[i] = (size_t)j;
            --skips;
          } else {
            ++skips;
            if (skips > max_skips) {
              stop = 2;
              break;
            }
          }
        }
        if (ctr) {
          uint64_t walked = (uint64_t)((int32_t)i - j - (stop ? 0 : 1));
          if (walked > ctr->longest_walk) ctr->longest_walk = walked;
          if (stop == 1) ctr->walks_target_gap++;
          if (stop == 2) ctr->walks_skips++;
          if (stop == 0 && start > 0) ctr->walks_band++;
          ctr->deep_link_ranges +=
              deep_link_range(A, i, band, max_target_gap_length, max_gap_length, qmin);
        }
        if (score[i] > gmax) gmax = score[i];
        if (score[i] >= min_score && score[i] > gmax / 2) {
          if (n_ends == cap_ends) {
            cap_ends *= 2;
            end_score = (float *)realloc(end_score, cap_ends * sizeof(float));
            end_idx = (size_t *)realloc(end_idx, cap_ends * sizeof(size_t));
          }
          end_score[n_ends] = score[i];
          end_idx[n_ends++] = i;
        }
      }
      /* :552-568: order (score desc, index desc); only the first 3 are ever used */
      unsigned char *taken = (unsigned char *)calloc(n_ends ? n_ends : 1, 1);
      for (int r = 0; r < num_best && (size_t)r < n_ends; ++r) {
        size_t best = (size_t)-1;
        for (size_t e = 0; e < n_ends; ++e) {
          if (taken[e]) continue;
          if (best == (size_t)-1 || end_score[e] > end_score[best] ||
              (end_score[e] == end_score[best] && end_idx[e] > end_idx[best]))
            best = e;
        }
        taken[best] = 1;
        if (ctr)
          for (size_t e = 0; e < n_ends; ++e)
            if (!taken[e] && end_score[e] == end_score[best]) {
              ctr->end_ties++;
              break;
            }
        /* direction_i == 0 -> Positive (dir 1) */
        traceback(s == 0 ? 1u : 0u, end_idx[best], (uint32_t)t, score, pred, A, used, chains, ctr);
        if (score[end_idx[best]] < gmax / 2) break;
      }
      free(taken);
      free(score);
      free(pred);
      free(used);
      free(end_score);
      free(end_idx);
    }
  }
  if (chains->n > 0) {
    /* :222-253 GeneratePrimaryChains: sort descending (insertion sort: total order) */
    for (size_t i = 1; i < chains->n; ++i) {
      orc_chain c = chains->chains[i];
      size_t j = i;
      while (j > 0 && chain_greater(&c, &chains->chains[j - 1])) {
        chains->chains[j] = chains->chains[j - 1];
        --j;
      }
      chains->chains[j] = c;
    }
    if (ctr)
      for (size_t i = 1; i < chains->n; ++i)
        ctr->primary_ties += chains->chains[i].score == chains->chains[i - 1].score;
    size_t np = 1;
    unsigned char *is_primary = (unsigned char *)calloc(chains->n, 1);
    size_t *prim = (size_t *)malloc(chains->n * sizeof(size_t));
    prim[0] = 0;
    is_primary[0] = 1;
    for (size_t ci = 1; ci < chains->n; ++ci) {
      const orc_chain *c = &chains->chains[ci];
      if (c->score < chains->chains[prim[np - 1]].score / 3) break;
      int ok = 1;
      for (size_t pi = 0; pi < np; ++pi) {
        const orc_chain *p = &chains->chains[prim[pi]];
        if (c->contig == p->contig) {
          uint32_t lo = c->start > p->start ? c->start : p->start;
          uint32_t hi = c->end < p->end ? c->end : p->end;
          if (!(lo > hi)) {
            ok = 0;
            break;
          }
        }
      }
      if (ok) {
        prim[np++] = ci;
        is_primary[ci] = 1;
      }
    }
    size_t k = 0;
    for (size_t ci = 0; ci < chains->n; ++ci) {
      if (is_primary[ci])
        chains->chains[k++] = chains->chains[ci];
      else
        free(chains->chains[ci].anchors);
    }
    chains->n = k;
    free(is_primary);
    free(prim);
    /* :255-274 ComputeMAPQ */
    if (chains->n == 1) {
      chains->chains[0].mapq = 60;
    } else {
      int mapq = (int)(40 * (1 - chains->chains[1].score / chains->chains[0].score));
      if (mapq > 60) mapq = 60;
      if (mapq < 0) mapq = 0;
      chains->chains[0].mapq = (uint32_t)(uint8_t)mapq;
    }
  }
}

static void seed_buckets(bucket *bk[2], size_t n_targets, orc_chain_list *chains) {
  for (int s = 0; s < 2; ++s) bk[s] = (bucket *)calloc(n_targets ? n_targets : 1, sizeof(bucket));
  /* spatial_index.cc:303-322: anchors of the previous chunk's chains go in first */
  for (size_t c = 0; c < chains->n; ++c) {
    int strand = chains->chains[c].dir == 1 ? 0 : 1;
    for (uint32_t a = 0; a < chains->chains[c].n_anchors; ++a)
      bucket_push(&bk[strand][chains->chains[c].contig], chains->chains[c].anchors[a]);
  }
  orc_chain_list_free(chains);
}

static void free_buckets(bucket *bk[2], size_t n_targets) {
  for (int s = 0; s < 2; ++s) {
    for (size_t t = 0; t < n_targets; ++t) free(bk[s][t].a);
    free(bk[s]);
  }
}

/* spatial_index.cc:371-402 */
static void emit_hit(bucket *bk[2], uint64_t P, uint32_t qpos, float d2) {
  uint32_t contig = (uint32_t)(P >> 33), tpos = (uint32_t)(P >> 1);
  int strand = (P & 1) == 0 ? 0 : 1;
  orc_anchor a = {tpos, qpos, d2};
  bucket_push(&bk[strand][contig], a);
}

void orc_generate_chains(const uint64_t *pos, const float *vals, size_t n_points,
                         const float *features, size_t n_features, uint32_t query_offset,
                         int step, float radius, size_t n_targets, orc_chain_list *chains) {
  orc_generate_chains_counted(pos, vals, n_points, features, n_features, query_offset, step,
                              radius, n_targets, chains, NULL);
}

void orc_generate_chains_counted(const uint64_t *pos, const float *vals, size_t n_points,
                                 const float *features, size_t n_features, uint32_t query_offset,
                                 int step, float radius, size_t n_targets, orc_chain_list *chains,
                                 orc_chain_counters *ctr) {
  const size_t num_nearest = 5000;
  bucket *bk[2];
  seed_buckets(bk, n_targets, chains);
  /* spatial_index.cc:326-409 with Q3: seeds at step, 2*step, ... */
  size_t np = n_features - DIM + 1;
  uint64_t *hi = (uint64_t *)malloc(num_nearest * sizeof(uint64_t));
  float *hd = (float *)malloc(num_nearest * sizeof(float));
  uint32_t prev = 0, count = 0;
  for (uint32_t p = 0; p < np; ++p) {
    if (p < prev + (uint32_t)step && p + (uint32_t)step > prev) continue;
    size_t nh = orc_radius_search(vals, n_points, features + p, radius, hi, hd, num_nearest);
    if (ctr && nh > ctr->max_query_hits) ctr->max_query_hits = nh;
    for (size_t a = 0; a < nh && a < num_nearest; ++a)
      emit_hit(bk, pos[hi[a]], p + query_offset, hd[a]);
    ++count;
    if (count >= np / (size_t)step) break;
    prev = p;
  }
  free(hi);
  free(hd);
  chain_buckets(bk, n_targets, radius, query_offset, chains, ctr);
  free_buckets(bk, n_targets);
}

void orc_chain_from_hits(const uint64_t *pos, const uint32_t *query_pos, size_t n_queries,
                         const uint64_t *hit_off, const uint64_t *hit_idx, const float *hit_d2,
                         float radius, size_t n_targets, orc_chain_list *chains) {
  bucket *bk[2];
  seed_buckets(bk, n_targets, chains);
  for (size_t k = 0; k < n_queries; ++k) {
    uint64_t n = hit_off[k + 1] - hit_off[k];
    for (uint64_t a = 0; a < n && a < 5000; ++a)
      emit_hit(bk, pos[hit_idx[hit_off[k] + a]], query_pos[k], hit_d2[hit_off[k] + a]);
  }
  chain_buckets(bk, n_targets, radius, 0, chains, NULL);
  free_buckets(bk, n_targets);
}

/* ------------------------------------------------------------------ A.4 */
void orc_streaming_map(const uint64_t *pos, const float *vals, size_t n_points,
                       size_t n_targets, const uint32_t *contig_len, const float *pa,
                       size_t n_pa, const orc_params *p, orc_mapping *out) {
  orc_streaming_map_counted(pos, vals, n_points, n_targets, contig_len, pa, n_pa, p, out, NULL);
}

void orc_streaming_map_counted(const uint64_t *pos, const float *vals, size_t n_points,
                               size_t n_targets, const uint32_t *contig_len, const float *pa,
                               size_t n_pa, const orc_params *p, orc_mapping *out,
                               orc_chain_counters *ctr) {
  const uint32_t bp_per_sec = 450, sample_rate = 4000, chunk_size = 4000;
  memset(out, 0, sizeof(*out));
  size_t num_chunks = n_pa / chunk_size;
  orc_chain_list chains = {NULL, 0, 0};
  uint32_t num_events = 0, ci = 0;
  float *feat = (float *)malloc((chunk_size + 2) * sizeof(float));
  for (ci = 0; ci < num_chunks && ci < (uint32_t)p->max_num_chunks; ++ci) {
    size_t nf = orc_generate_events(pa + (size_t)chunk_size * ci, chunk_size, feat);
    if (nf > 50) {
      orc_generate_chains_counted(pos, vals, n_points, feat, nf, num_events, p->step,
                                  p->search_radius, n_targets, &chains, ctr);
      num_events += (uint32_t)nf;
      if (chains.n >= 2) {
        if (chains.chains[0].score / chains.chains[1].score >= p->stop_ratio) break;
        float mean = 0;
        for (size_t c = 0; c < chains.n; ++c) mean += chains.chains[c].score;
        mean /= chains.n;
        if (chains.chains[0].score >= p->stop_mean_ratio * mean) break;
      } else if (chains.n == 1 && chains.chains[0].n_anchors >= (uint32_t)p->stop_min_anchors) {
        break;
      }
    }
  }
  free(feat);
  if (ci > 0 && (ci == num_chunks || ci == (uint32_t)p->max_num_chunks)) --ci;
  float scale = ((float)(ci + 1) * chunk_size / num_events) / ((float)sample_rate / bp_per_sec);
  float mean = 0;
  for (size_t c = 0; c < chains.n; ++c) mean += chains.chains[c].score;
  mean /= chains.n;
  out->read_len = (uint32_t)n_pa;
  out->chunks = ci + 1;
  out->n_chains = (uint32_t)chains.n;
  out->num_events = num_events;
  out->mapq = 61;
  if (chains.n >= 1) {
    const orc_chain *c0 = &chains.chains[0];
    float ad = 0, at = 0, aq = 0;
    for (size_t ai = 0; ai < c0->n_anchors; ++ai) {
      ad += c0->anchors[ai].dist;
      if (ai + 1 < c0->n_anchors) {
        at += (float)(uint32_t)(c0->anchors[ai].target - c0->anchors[ai + 1].target);
        aq += (float)(uint32_t)(c0->anchors[ai].query - c0->anchors[ai + 1].query);
      }
    }
    ad /= c0->n_anchors;
    at /= c0->n_anchors;
    aq /= c0->n_anchors;
    out->cm = c0->n_anchors;
    out->s1 = c0->score;
    out->s2 = chains.n > 1 ? chains.chains[1].score : 0;
    out->sm = mean;
    out->ad = ad;
    out->at = at;
    out->aq = aq;
    int mapped =
        (chains.n >= 2 && (c0->score / chains.chains[1].score >= p->output_ratio ||
                           c0->score >= p->output_mean_ratio * mean)) ||
        (chains.n == 1 && c0->n_anchors >= (uint32_t)p->output_min_anchors);
    if (mapped) {
      out->mapped = 1;
      out->q_start = (uint32_t)(scale * c0->anchors[c0->n_anchors - 1].query);
      out->q_end = (uint32_t)(scale * c0->anchors[0].query);
      out->strand_plus = c0->dir;
      out->contig = c0->contig;
      out->t_start = c0->dir == 1 ? c0->start : (uint32_t)(contig_len[c0->contig] + 1 - c0->end);
      out->frag_len = c0->end - c0->start + 1;
      out->mapq = c0->mapq & 63u; /* 6-bit field, output_tools.h:24 */
    }
  }
  orc_chain_list_free(&chains);
}

int orc_format_paf(const orc_mapping *m, const char *read_name, const char *contig_name,
                   uint32_t contig_len, double mt_ms, char *buf, size_t cap) {
  char tags[512];
  int k = snprintf(tags, sizeof tags, "mt:f:%f\tci:i:%u\tsl:i:%u", mt_ms, m->chunks, m->read_len);
  if (m->n_chains >= 1)
    k += snprintf(tags + k, sizeof tags - k,
                  "\tcm:i:%u\tnc:i:%u\ts1:f:%f\ts2:f:%f\tsm:f:%f\tad:f:%f\tat:f:%f\taq:f:%f", m->cm,
                  m->n_chains, (double)m->s1, (double)m->s2, (double)m->sm, (double)m->ad,
                  (double)m->at, (double)m->aq);
  if (m->mapped && m->mapq <= 60)
    return snprintf(buf, cap, "%s\t%u\t%u\t%u\t%s\t%s\t%u\t%u\t%u\t%u\t%u\t%u\t%s\n", read_name,
                    m->read_len, m->q_start, m->q_end, m->strand_plus ? "+" : "-", contig_name,
                    contig_len, m->t_start, m->t_start + m->frag_len, m->read_len, m->frag_len,
                    m->mapq, tags);
  return snprintf(buf, cap, "%s\t%u\t*\t*\t*\t*\t*\t*\t*\t*\t*\t%u\t%s\n", read_name, m->read_len,
                  61u, tags);
}

/* ------------------------------------------------------------------ A.5 */
static const unsigned char base_code[256] = {
    ['A'] = 1, ['C'] = 2, ['G'] = 3, ['T'] = 4, ['a'] = 1, ['c'] = 2, ['g'] = 3, ['t'] = 4};
static inline int code_of(char c) { return (int)base_code[(unsigned char)c] - 1; } /* -1: ambiguous */

/* pore_model.cc:57-80 with the off-by-one of Q1; seq must be NUL-terminated */
static void level_means(const char *seq, uint32_t len, const float *level_mean, float *out) {
  int32_t L = (int32_t)len - 6 + 1;
  uint32_t mask = (1u << 12) - 1, h = 0;
  for (uint32_t i = 0; i < 6; ++i) { /* utils.h GenerateSeedFromSequence, sequence_length = L */
    if (i < (uint32_t)L) {
      int c = code_of(seq[i]);
      h = c >= 0 ? (((h << 2) | (uint32_t)c) & mask) : ((h << 2) & mask);
    } else {
      h = (h << 2) & mask;
    }
  }
  out[0] = level_mean[h];
  for (uint32_t p = 1; p < len - 6 + 1; ++p) {
    int c = code_of(seq[p + 6]); /* Q1: reads one base too far; seq[len] is NUL -> 'A' */
    h = c >= 0 ? (((h << 2) | (uint32_t)c) & mask) : ((h << 2) & mask);
    out[p] = level_mean[h];
  }
}

static void revcomp(const char *s, uint32_t len, char *out) { /* sequence_batch.h:66-77 */
  static const char tab[5] = {'A', 'C', 'G', 'T', 'N'};
  for (uint32_t i = 0; i < len; ++i) {
    int c = code_of(s[len - i - 1]);
    out[i] = c >= 0 ? tab[3 ^ c] : 'N'; /* Uint8ToChar(3 ^ 4 = 7) = 'N' */
  }
  out[len] = 0;
}

/* sigmap.cc:19-185 with k = 11: direct-addressed counts replace the khash */
static void kmer_pass(const char *seq, uint32_t len, int k, uint32_t *hist, uint64_t *num_kmers,
                      unsigned char *mask_out, float frequency) {
  uint64_t shift = 2 * (uint64_t)(k - 1), m = ((uint64_t)1 << (2 * k)) - 1, f = 0, r = 0;
  int unamb = 0;
  for (uint32_t p = 0; p < len; ++p) {
    int c = code_of(seq[p]);
    if (c >= 0) {
      f = ((f << 2) | (uint64_t)c) & m;
      r = (r >> 2) | ((uint64_t)(3 ^ c) << shift);
      ++unamb;
      if (unamb >= k) {
        uint64_t canon = f < r ? f : r;
        if (!mask_out) {
          hist[canon]++;
          ++*num_kmers;
        } else {
          float fr = (float)hist[canon] / (float)*num_kmers;
          mask_out[p + 1 - k] = fr > frequency;
        }
      }
    } else {
      unamb = 0;
      f = r = 0;
      if (mask_out && p >= (uint32_t)k - 1) mask_out[p + 1 - k] = 1;
    }
  }
}

size_t orc_build_point_cloud(const char *const *seqs, const uint32_t *seq_len, size_t n_seq,
                             const float *level_mean, uint64_t *pos, float *vals) {
  const int k = DIM + 6 - 1; /* sigmap.cc:1014 */
  uint32_t *hist = (uint32_t *)calloc((size_t)1 << (2 * k), sizeof(uint32_t));
  uint64_t num_kmers = 0;
  for (size_t s = 0; s < n_seq; ++s) kmer_pass(seqs[s], seq_len[s], k, hist, &num_kmers, NULL, 0);
  size_t n = 0;
  float last_value = 0;
  int have_last = 0;
  for (int strand = 0; strand < 2; ++strand) { /* spatial_index.cc:82-93: all +, then all - */
    for (size_t s = 0; s < n_seq; ++s) {
      uint32_t len = seq_len[s];
      char *neg = NULL;
      const char *seq = seqs[s];
      if (strand == 1) {
        neg = (char *)malloc((size_t)len + 1);
        revcomp(seqs[s], len, neg);
        seq = neg;
      }
      uint32_t L = len - 6 + 1;
      float *lv = (float *)malloc(L * sizeof(float));
      float *z = (float *)malloc(L * sizeof(float));
      level_means(seq, len, level_mean, lv);
      zscore(lv, L, z);
      unsigned char *masked = (unsigned char *)calloc(len - k + 1, 1);
      kmer_pass(seq, len, k, hist, &num_kmers, masked, 0.0002f);
      if (L >= DIM) {
        for (uint32_t p = 0; p < L - DIM + 1; ++p) { /* spatial_index.cc:39-56 */
          if (masked[p]) continue;
          if (p == 0 || !have_last || fabs((double)(z[p] - last_value)) > 0.01) {
            if (pos) {
              pos[n] = ((((uint64_t)s) << 32 | p) << 1) | (uint64_t)strand;
              vals[n] = z[p];
            }
            last_value = z[p];
            have_last = 1;
            ++n;
          }
        }
      }
      free(masked);
      free(lv);
      free(z);
      free(neg);
    }
  }
  free(hist);
  return n;
}
