// k_events.cuh -- K1 (raw -> pA filter + compaction) and K2/K3 (event detection,
// z-normalisation, compression) for a batch of 4000-sample chunks.
//
// Bit-faithful to the reference's strict-FP build (SURVEY.md H1/H2, Appendix A.0/A.1):
//   * the fp32 prefix sums are SEQUENTIAL per chunk (event.h:64-67) -- a parallel scan
//     changes fp32 rounding and costs ~1 % of PAF rows -- so the sequential stages run one
//     THREAD per chunk, and every per-sample array is stored TRANSPOSED ([sample][chunk])
//     so the 32 lanes of a warp (32 different chunks) read/write one coalesced 128-byte
//     line per step;
//   * the t-statistics (embarrassingly parallel, fp64 sqrt/div as in event.h:109, Q6) run
//     one thread per (chunk, strip of samples) at full occupancy;
//   * the coupled two-detector peak state machine (event.h:117-182) is inherently
//     sequential: one thread per chunk again, t-stats prefetched 8 steps ahead.
// No FMA anywhere (-fmad=false), IEEE division and square root.
#ifndef SB_K_EVENTS_CUH
#define SB_K_EVENTS_CUH

#include <float.h>

#include "sb_device.cuh"

namespace sb {

// ---------------------------------------------------------------- K1
// One block per read.  pA = (float(raw) + offset) * (range / digitisation); keep iff
// 30 < pA < 200 (signal_batch.cc:196-207).  Kept RAW samples are compacted (order kept)
// to kept + kept_off[r]; the events kernel redoes the identical conversion.
// Read r is raw[read_beg[r] .. read_end[r]): reads packed end to end pass read_off and
// read_off + 1, reads anywhere in a caller's device buffer a start and an end table.
constexpr int kFilterThreads = 256;
constexpr int kFilterPerThread = 8;

__device__ __forceinline__ float raw_to_pa(int16_t raw, float offset, float scale) {
  return __fmul_rn(__fadd_rn((float)raw, offset), scale);
}

__global__ void __launch_bounds__(kFilterThreads)
k_filter_compact(const int16_t *__restrict__ raw, const uint64_t *__restrict__ read_beg,
                 const uint64_t *__restrict__ read_end,
                 const float *__restrict__ dig, const float *__restrict__ range,
                 const float *__restrict__ offset, const uint64_t *__restrict__ kept_off,
                 int16_t *__restrict__ kept, uint32_t *__restrict__ kept_len, uint32_t n_reads) {
  const uint32_t r = blockIdx.x;
  if (r >= n_reads) return;
  const uint64_t beg = read_beg[r], n = read_end[r] - beg;
  const float off = offset[r], scale = __fdiv_rn(range[r], dig[r]);
  int16_t *out = kept + kept_off[r];
  __shared__ uint32_t warp_tot[kFilterThreads / 32];
  __shared__ uint32_t tile_tot;
  uint64_t written = 0;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (uint64_t tile = 0; tile < n; tile += kFilterThreads * kFilterPerThread) {
    const uint64_t s0 = tile + (uint64_t)threadIdx.x * kFilterPerThread;
    int16_t v[kFilterPerThread];
    uint32_t keep = 0;
#pragma unroll
    for (int k = 0; k < kFilterPerThread; ++k) {
      v[k] = 0;
      if (s0 + k < n) {
        v[k] = raw[beg + s0 + k];
        float pa = raw_to_pa(v[k], off, scale);
        if (pa > 30.0f && pa < 200.0f) keep |= 1u << k;
      }
    }
    const uint32_t cnt = __popc(keep);
    uint32_t incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t acc = 0;
      for (int w = 0; w < kFilterThreads / 32; ++w) {
        uint32_t t = warp_tot[w];
        warp_tot[w] = acc;
        acc += t;
      }
      tile_tot = acc;
    }
    __syncthreads();
    uint64_t dst = written + warp_tot[wid] + (incl - cnt);
#pragma unroll
    for (int k = 0; k < kFilterPerThread; ++k)
      if (keep & (1u << k)) out[dst++] = v[k];
    written += tile_tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) kept_len[r] = (uint32_t)written;
}

// kept raw -> pA floats (stage hook only)
__global__ void k_raw_to_pa(const int16_t *__restrict__ kept, uint32_t n, float offset, float scale,
                            float *__restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = raw_to_pa(kept[i], offset, scale);
}

// ---------------------------------------------------------------- K2a: sequential prefix sums
// Thread b scans chunk b.  ps/pss are [kChunk+1][Bp] (transposed).  RAW=true: input is the
// compacted int16 stream (16-byte aligned chunk starts); RAW=false: fp32 pA (stage hook).
template <bool RAW>
__global__ void __launch_bounds__(128)
k_ev_prefix(const void *__restrict__ src, const uint64_t *__restrict__ chunk_start,
            const float *__restrict__ chunk_offset, const float *__restrict__ chunk_scale,
            float *__restrict__ ps, float *__restrict__ pss, uint32_t B, uint32_t Bp) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float s = 0.0f, q = 0.0f;
  ps[b] = 0.0f;
  pss[b] = 0.0f;
  size_t o = (size_t)Bp + b;
  if (RAW) {
    const int4 *in = reinterpret_cast<const int4 *>(static_cast<const int16_t *>(src) + chunk_start[b]);
    const float off = chunk_offset[b], scale = chunk_scale[b];
#pragma unroll 2
    for (int i = 0; i < kChunk / 8; ++i) {
      int4 w = __ldg(in + i);
      __align__(16) int16_t v[8];
      *reinterpret_cast<int4 *>(v) = w;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float x = raw_to_pa(v[k], off, scale);
        s = __fadd_rn(s, x);
        q = __fadd_rn(q, __fmul_rn(x, x));
        ps[o] = s;
        pss[o] = q;
        o += Bp;
      }
    }
  } else {
    const float4 *in = reinterpret_cast<const float4 *>(static_cast<const float *>(src) + chunk_start[b]);
#pragma unroll 2
    for (int i = 0; i < kChunk / 4; ++i) {
      float4 w = __ldg(in + i);
      float v[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float x = v[k];
        s = __fadd_rn(s, x);
        q = __fadd_rn(q, __fmul_rn(x, x));
        ps[o] = s;
        pss[o] = q;
        o += Bp;
      }
    }
  }
}

// ---------------------------------------------------------------- K2b: t-statistics
// event.h:70-115 for w = 3 and w = 6.  Thread = (chunk b, strip of kStrip sample indices).
constexpr int kStrip = 16;

__device__ __forceinline__ float tstat_at(const float *p, const float *q, int c, int w) {
  // p/q are register windows; index c is position i, window half-width w
  const float wf = (float)w;
  float sum1 = __fsub_rn(p[c], p[c - w]);       // ps[i-w] = 0 when i == w, so this is exact
  float sumsq1 = __fsub_rn(q[c], q[c - w]);
  float sum2 = __fsub_rn(p[c + w], p[c]);
  float sumsq2 = __fsub_rn(q[c + w], q[c]);
  float mean1 = __fdiv_rn(sum1, wf), mean2 = __fdiv_rn(sum2, wf);
  float cv = __fsub_rn(__fadd_rn(__fsub_rn(__fdiv_rn(sumsq1, wf), __fmul_rn(mean1, mean1)),
                                 __fdiv_rn(sumsq2, wf)),
                       __fmul_rn(mean2, mean2));
  cv = fmaxf(cv, FLT_MIN);
  float dm = __fsub_rn(mean2, mean1);
  float cvw = __fdiv_rn(cv, wf);
  return (float)__ddiv_rn(fabs((double)dm), __dsqrt_rn((double)cvw));  // Q6: binary64
}

__global__ void __launch_bounds__(128)
k_ev_tstat(const float *__restrict__ ps, const float *__restrict__ pss, float *__restrict__ t1,
           float *__restrict__ t2, uint32_t B, uint32_t Bp) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int i0 = blockIdx.y * kStrip;  // outputs i0 .. i0+kStrip-1, i in [0, kChunk]
  float p[kStrip + 12], q[kStrip + 12];
#pragma unroll
  for (int k = 0; k < kStrip + 12; ++k) {
    int i = i0 - 6 + k;
    bool ok = i >= 0 && i <= kChunk;
    p[k] = ok ? __ldg(ps + (size_t)i * Bp + b) : 0.0f;
    q[k] = ok ? __ldg(pss + (size_t)i * Bp + b) : 0.0f;
  }
#pragma unroll
  for (int k = 0; k < kStrip; ++k) {
    int i = i0 + k;
    if (i > kChunk) break;
    // zeros on [0,w) and (n-w, n]  (event.h:85-87,112-114)
    float a = (i >= 3 && i <= kChunk - 3) ? tstat_at(p, q, k + 6, 3) : 0.0f;
    float c = (i >= 6 && i <= kChunk - 6) ? tstat_at(p, q, k + 6, 6) : 0.0f;
    t1[(size_t)i * Bp + b] = a;
    t2[(size_t)i * Bp + b] = c;
  }
}

// ---------------------------------------------------------------- K2c/K3: peaks -> events -> features
// Thread b: the two-detector state machine over t1/t2 (event.h:117-182), event means from the
// prefix sums (event.h:184-224), z-score with double accumulators (sigmap.cc:1131-1155) and
// the |dz| > 0.1 compression (sigmap.cc:1073-1079).  means/features are chunk-major scratch
// rows of kFeatCap floats.
struct Det {
  float thr, peak_value;
  int w, peak_pos, masked_to;  // masked_to: size_t in the reference, never exceeds n + w
  bool valid;
};

// Where the detector reads its per-sample inputs: the transposed global arrays of the
// thread-per-chunk path, or the shared-memory rows of the warp-per-chunk path.
struct EvGlobalSrc {
  const float *t1, *t2, *ps;
  uint32_t Bp, b;
  __device__ __forceinline__ void load8(int base, float *a, float *c) const {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      a[k] = __ldg(t1 + (size_t)(base + k) * Bp + b);
      c[k] = __ldg(t2 + (size_t)(base + k) * Bp + b);
    }
  }
  __device__ __forceinline__ float prefix(unsigned long long i) const { return __ldg(ps + (size_t)i * Bp + b); }
};
struct EvSharedSrc {
  const float *t1, *t2, *ps;
  __device__ __forceinline__ void load8(int base, float *a, float *c) const {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      a[k] = t1[base + k];
      c[k] = t2[base + k];
    }
  }
  __device__ __forceinline__ float prefix(unsigned long long i) const { return ps[i]; }
};

// One thread, one chunk: peaks -> events -> z-scores -> compressed features.
template <class Src>
__device__ __forceinline__ void ev_detect_features(const Src &src, float *__restrict__ my_means,
                                                   float *__restrict__ my_feat,
                                                   uint32_t *__restrict__ my_peaks /* optional */,
                                                   uint32_t &nf_out, uint32_t &ne_out) {
  Det sd = {4.30265f, FLT_MAX, 3, -1, 0, false};  // event.h:31-37 defaults
  Det ld = {2.57058f, FLT_MAX, 6, -1, 0, false};
  const float peak_height = 1.0f;
  uint32_t np = 0;
  int prev_peak = 0, prev_prev_peak = 0;
  auto emit = [&](int pos) {
    // event k = (peaks[k-1], peaks[k]) (k = 0: start 0); the LAST peak's event is replaced below
    if (np < (uint32_t)kFeatCap) {
      unsigned long long s = np == 0 ? 0ull : (unsigned long long)prev_peak;
      unsigned long long len = (unsigned long long)pos - s;  // unsigned wrap as in the reference
      float d = __fsub_rn(src.prefix((unsigned long long)pos), src.prefix(s));
      my_means[np] = __fdiv_rn(d, (float)len);
      if (my_peaks) my_peaks[np] = (uint32_t)pos;
    }
    prev_prev_peak = prev_peak;
    prev_peak = pos;
    ++np;
  };
  for (int base = 0; base < kChunk; base += 8) {
    float a[8], c[8];
    src.load8(base, a, c);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int i = base + k;
      // ---- short detector
      if (sd.masked_to < i) {
        const float cur = a[k];
        if (sd.peak_pos == -1) {
          if (cur < sd.peak_value) {
            sd.peak_value = cur;
          } else if (__fsub_rn(cur, sd.peak_value) > peak_height) {
            sd.peak_value = cur;
            sd.peak_pos = i;
          }
        } else {
          if (cur > sd.peak_value) {
            sd.peak_value = cur;
            sd.peak_pos = i;
          }
          if (sd.peak_value > sd.thr) {  // short dominates long (event.h:156-164)
            ld.masked_to = sd.peak_pos + sd.w;
            ld.peak_pos = -1;
            ld.peak_value = FLT_MAX;
            ld.valid = false;
          }
          if (__fsub_rn(sd.peak_value, cur) > peak_height && sd.peak_value > sd.thr) sd.valid = true;
          if (sd.valid && (i - sd.peak_pos) > sd.w / 2) {
            emit(sd.peak_pos);
            sd.peak_pos = -1;
            sd.peak_value = cur;
            sd.valid = false;
          }
        }
      }
      // ---- long detector
      if (ld.masked_to < i) {
        const float cur = c[k];
        if (ld.peak_pos == -1) {
          if (cur < ld.peak_value) {
            ld.peak_value = cur;
          } else if (__fsub_rn(cur, ld.peak_value) > peak_height) {
            ld.peak_value = cur;
            ld.peak_pos = i;
          }
        } else {
          if (cur > ld.peak_value) {
            ld.peak_value = cur;
            ld.peak_pos = i;
          }
          if (__fsub_rn(ld.peak_value, cur) > peak_height && ld.peak_value > ld.thr) ld.valid = true;
          if (ld.valid && (i - ld.peak_pos) > ld.w / 2) {
            emit(ld.peak_pos);
            ld.peak_pos = -1;
            ld.peak_value = cur;
            ld.valid = false;
          }
        }
      }
    }
  }
  // CreateEvents (event.h:200-224): ne = #peaks events; the last one runs (peaks[ne-2], n).
  // Fewer than two peaks is undefined behaviour in the reference -> no events here.
  uint32_t ne = (np >= 2 && np <= (uint32_t)kFeatCap) ? np : 0;
  uint32_t nf = 0;
  if (ne) {
    {
      unsigned long long s = (unsigned long long)prev_prev_peak;  // peaks[ne-2]
      unsigned long long len = (unsigned long long)kChunk - s;
      float d = __fsub_rn(src.prefix((unsigned long long)kChunk), src.prefix(s));
      my_means[ne - 1] = __fdiv_rn(d, (float)len);
    }
    double mean = 0.0;
    for (uint32_t k = 0; k < ne; ++k) mean = __dadd_rn(mean, (double)my_means[k]);
    mean = __ddiv_rn(mean, (double)ne);
    double ss = 0.0;
    for (uint32_t k = 0; k < ne; ++k) {
      double d = __dsub_rn((double)my_means[k], mean);
      ss = __dadd_rn(ss, __dmul_rn(d, d));
    }
    const double sdv = __dsqrt_rn(__ddiv_rn(ss, (double)(ne - 1)));
    float last = 0.0f;
    for (uint32_t k = 0; k < ne; ++k) {
      float z = (float)__ddiv_rn(__dsub_rn((double)my_means[k], mean), sdv);
      if (k == 0 || (double)fabsf(__fsub_rn(z, last)) > 0.1) {  // Q5: float abs vs double 0.1
        my_feat[nf++] = z;
        last = z;
      }
    }
  }
  nf_out = nf;
  ne_out = ne;
}

__global__ void __launch_bounds__(128)
k_ev_features(const float *__restrict__ t1, const float *__restrict__ t2,
              const float *__restrict__ ps, float *__restrict__ means, float *__restrict__ features,
              uint32_t *__restrict__ n_features, uint32_t *__restrict__ n_raw_events,
              uint32_t *__restrict__ peaks_out /* optional, chunk-major kFeatCap */, uint32_t B,
              uint32_t Bp, Counters *__restrict__ ctr) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const EvGlobalSrc src{t1, t2, ps, Bp, b};
  uint32_t nf = 0, ne = 0;
  ev_detect_features(src, means + (size_t)b * kFeatCap, features + (size_t)b * kFeatCap,
                     peaks_out ? peaks_out + (size_t)b * kFeatCap : nullptr, nf, ne);
  n_features[b] = nf;
  if (n_raw_events) n_raw_events[b] = ne;
  if (ctr) {
    atomicAdd(&ctr->n_events_raw, (unsigned long long)ne);
    atomicAdd(&ctr->n_events_kept, (unsigned long long)nf);
  }
}

// ---------------------------------------------------------------- small batches: warp per chunk
// The read-until path maps a few hundred chunks per round; with one THREAD per chunk that is a
// handful of warps whose 32 lanes diverge through the detector and wait on global memory every
// step.  Here one WARP owns a chunk and keeps it in shared memory: all lanes load and convert
// the samples and compute the t-statistics; the two order-dependent parts (the fp32 prefix sums
// and the detector / z-score / compression tail) run on lane 0 alone with the same expressions
// as the thread-per-chunk kernels, so results are bit-identical.
//   rows: ps[0..4000], pss[0..4000] (overwritten in place by t2, one tile behind), t1[0..4000]
constexpr int kEvRow = kChunk + 8;  // floats per shared row (16-byte multiple)
constexpr size_t kEvWarpSmem = (size_t)3 * kEvRow * sizeof(float);

template <bool RAW>
__global__ void __launch_bounds__(32)
k_ev_chunk_warp(const void *__restrict__ src, const uint64_t *__restrict__ chunk_start,
                const float *__restrict__ chunk_offset, const float *__restrict__ chunk_scale,
                float *__restrict__ means, float *__restrict__ features,
                uint32_t *__restrict__ n_features, uint32_t *__restrict__ n_raw_events,
                uint32_t *__restrict__ peaks_out /* optional */, uint32_t B,
                Counters *__restrict__ ctr) {
  extern __shared__ __align__(16) float s_ev[];
  const uint32_t b = blockIdx.x;
  if (b >= B) return;
  const int lane = threadIdx.x;
  float *ps = s_ev, *pss = s_ev + kEvRow, *t1 = s_ev + 2 * kEvRow;
  // ---- samples -> ps[i+1] = x_i, pss[i+1] = x_i * x_i (all lanes)
  if (RAW) {
    const int4 *in = reinterpret_cast<const int4 *>(static_cast<const int16_t *>(src) + chunk_start[b]);
    const float off = chunk_offset[b], scale = chunk_scale[b];
    for (int i = lane; i < kChunk / 8; i += 32) {
      const int4 w = __ldg(in + i);
      __align__(16) int16_t v[8];
      *reinterpret_cast<int4 *>(v) = w;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float x = raw_to_pa(v[k], off, scale);
        ps[1 + 8 * i + k] = x;
        pss[1 + 8 * i + k] = __fmul_rn(x, x);
      }
    }
  } else {
    const float4 *in = reinterpret_cast<const float4 *>(static_cast<const float *>(src) + chunk_start[b]);
    for (int i = lane; i < kChunk / 4; i += 32) {
      const float4 w = __ldg(in + i);
      const float v[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        ps[1 + 4 * i + k] = v[k];
        pss[1 + 4 * i + k] = __fmul_rn(v[k], v[k]);
      }
    }
  }
  __syncwarp();
  // ---- sequential fp32 prefix sums, in place (event.h:58-68)
  if (lane == 0) {
    float s = 0.0f, q = 0.0f;
    ps[0] = 0.0f;
    pss[0] = 0.0f;
    for (int i = 1; i <= kChunk; i += 8) {
      float x[8], y[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        x[k] = ps[i + k];
        y[k] = pss[i + k];
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        s = __fadd_rn(s, x[k]);
        q = __fadd_rn(q, y[k]);
        ps[i + k] = s;
        pss[i + k] = q;
      }
    }
  }
  __syncwarp();
  // ---- t-statistics, 32 positions per tile; t2 replaces pss one tile behind the reads
  {
    float held = 0.0f;
    int held_i = -1;
    for (int base = 0; base <= kChunk; base += 32) {
      const int i = base + lane;
      float a = 0.0f, c = 0.0f;
      if (i <= kChunk) {
        // zeros on [0,w) and (n-w, n]  (event.h:85-87,112-114)
        if (i >= 3 && i <= kChunk - 3) a = tstat_at(ps, pss, i, 3);
        if (i >= 6 && i <= kChunk - 6) c = tstat_at(ps, pss, i, 6);
      }
      __syncwarp();  // this tile's reads of pss[base-6 .. base+37] are done
      if (held_i >= 0) pss[held_i] = held;  // previous tile: [base-32, base)
      if (i <= kChunk) {
        t1[i] = a;
        held = c;
        held_i = i;
      } else {
        held_i = -1;
      }
      __syncwarp();
    }
    if (held_i >= 0) pss[held_i] = held;
    __syncwarp();
  }
  // ---- detector and tail on lane 0
  if (lane == 0) {
    const EvSharedSrc ssrc{t1, pss, ps};
    uint32_t nf = 0, ne = 0;
    ev_detect_features(ssrc, means + (size_t)b * kFeatCap, features + (size_t)b * kFeatCap,
                       peaks_out ? peaks_out + (size_t)b * kFeatCap : nullptr, nf, ne);
    n_features[b] = nf;
    if (n_raw_events) n_raw_events[b] = ne;
    if (ctr) {
      atomicAdd(&ctr->n_events_raw, (unsigned long long)ne);
      atomicAdd(&ctr->n_events_kept, (unsigned long long)nf);
    }
  }
}

}  // namespace sb
#endif
