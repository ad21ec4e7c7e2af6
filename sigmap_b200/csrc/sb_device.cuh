// sb_device.cuh -- shared device-side definitions of the B200 mapping engine.
//
// Everything here is compiled for sm_100a only, with -fmad=false: the event features must
// reproduce the reference's strict IEEE fp32/fp64 arithmetic bit for bit (SURVEY.md H1), so
// no multiply-add contraction is allowed anywhere in this library.
#ifndef SB_DEVICE_CUH
#define SB_DEVICE_CUH

#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "../../include/sigmap_b200.h"

namespace sb {

constexpr int kChunk = SMB_CHUNK;       // 4000 samples
constexpr int kDim = SMB_DIM;           // 6
constexpr int kFeatCap = SMB_CHUNK;     // per-chunk event/feature capacity (peaks < samples)
constexpr int kMinFeatures = 50;        // sigmap.cc:660: GenerateChains only if size() > 50
constexpr uint32_t kMaxHits = SMB_MAX_HITS;
constexpr int kLeaf = 8;                // points per leaf = one 8-lane group (32-byte sectors)
constexpr int kFan = 8;                 // children per node; a warp tests 4 nodes per step
constexpr int kMaxLevels = 12;          // 8^12 leaves: never reached below 2^32 points

// cudaFree waits for the whole device -- including an upload still queued on the copy stream,
// which would serialise the upload and the mapping it is supposed to hide behind.  While a
// mapping call's DeferFrees (sb_engine.cu) is alive, buffers that have to grow park their old
// allocation here; it is released when the call's mapping is over (after a failure, cudaFree then
// waits for whatever the call left queued).
struct FreeLater {
  static inline thread_local bool on = false;
  static inline thread_local std::vector<void *> parked;
  static void drain() {
    for (void *q : parked) cudaFree(q);
    parked.clear();
  }
};
inline void dev_free(void *q) {
  if (FreeLater::on) FreeLater::parked.push_back(q);
  else cudaFree(q);
}

struct DeviceMem {
  static cudaError_t alloc(void **q, size_t bytes) { return cudaMalloc(q, bytes); }
  static void free(void *q) { dev_free(q); }
};
struct PinnedMem {
  static cudaError_t alloc(void **q, size_t bytes) { return cudaMallocHost(q, bytes); }
  static void free(void *q) { cudaFreeHost(q); }
};

// An array that frees itself: device memory (DevBuf) or pinned host memory (PinnedBuf).  Move-only.
// The destructor frees on the current device, so an owner must be destroyed with its context's
// device current: every entry point calls cudaSetDevice first, and smb_destroy / smb_batch_destroy
// do so before they delete.  cudaFree waits for the work queued on the device, so a buffer that goes
// out of scope on an error return waits for that work as an explicit release() would.
template <class T, class Mem>
struct Buf {
  T *p = nullptr;
  size_t cap = 0;  // elements
  Buf() = default;
  Buf(const Buf &) = delete;
  Buf &operator=(const Buf &) = delete;
  Buf(Buf &&o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
  Buf &operator=(Buf &&o) noexcept {
    if (this != &o) {
      release();
      p = std::exchange(o.p, nullptr);
      cap = std::exchange(o.cap, 0);
    }
    return *this;
  }
  ~Buf() { release(); }
  // at least n elements, with room to grow (contents are NOT preserved across growth)
  cudaError_t ensure(size_t n) {
    if (n <= cap) return cudaSuccess;
    const size_t want = n + n / 4 + 64;
    return take(want, want);
  }
  // exactly n elements (one when n = 0, so that p is a valid pointer)
  cudaError_t alloc(size_t n) { return take(std::max<size_t>(n, 1), n); }
  void release() {
    if (p) Mem::free(p);
    p = nullptr;
    cap = 0;
  }

 private:
  cudaError_t take(size_t elems, size_t n) {
    release();
    const cudaError_t e = Mem::alloc((void **)&p, elems * sizeof(T));
    if (e != cudaSuccess) {
      p = nullptr;
      cudaGetLastError();  // an out-of-memory return is not sticky: clear it, or the next launch check reports it
      return e;
    }
    cap = n;
    return e;
  }
};
template <class T>
using DevBuf = Buf<T, DeviceMem>;
template <class T>
using PinnedBuf = Buf<T, PinnedMem>;

// A stream or an event that destroys itself.  Create it with cudaStreamCreate*(&s.h) /
// cudaEventCreate*(&e.h); it converts to the raw handle.  Same device rule as Buf.
template <class H, cudaError_t (*Destroy)(H)>
struct Handle {
  H h = nullptr;
  Handle() = default;
  Handle(const Handle &) = delete;
  Handle &operator=(const Handle &) = delete;
  Handle(Handle &&o) noexcept : h(std::exchange(o.h, nullptr)) {}
  ~Handle() {
    if (h) Destroy(h);
  }
  operator H() const { return h; }
};
using Stream = Handle<cudaStream_t, cudaStreamDestroy>;
using Event = Handle<cudaEvent_t, cudaEventDestroy>;

// ---- flat device index over the ordered window points (replaces nanoflann) ----
// Leaves hold 8 consecutive points of the point order (aligned KD order, k_index.cuh); a node
// holds the boxes of its 8 children (level 0: leaves 8n..8n+7, level l: nodes 8n..8n+7 of level
// l-1), pointer-free.
// A warp works on FOUR nodes (or leaves) per half step, one 8-lane group each, so records are
// laid out for 8 lanes:
//   node  = [3][8 children] x four binary16: (lo0 lo1 lo2 lo3) (lo4 lo5 hi0 hi1) (hi2 hi3 hi4 hi5),
//           box corners rounded outwards, 192 bytes, three coalesced 64-byte loads per lane group;
//   leaf  = [3][8 points] float2 (v0 v1) (v2 v3) (v4 v5), then [8] {target, bucket}: 256 bytes.
//           The payload of a hit sits in the record the hit lane has just read (same 256-byte
//           block), so emitting an anchor costs no dependent random load.
// All node levels live in ONE buffer, top level first: the prefix that fits 64 KB (the levels
// every query walks) is staged in shared memory by the search kernel with one TMA bulk copy.
constexpr int kNodeRec = 3 * kFan;       // uint2 per node record
constexpr int kLeafRec = 4 * kLeaf;      // uint2 per leaf record (24 values + 8 payload)
constexpr uint32_t kTopSmemMax = 64u << 10;
constexpr float kPadValue = 1.0e18f;  // padding points: never inside any ball
struct IndexView {
  uint64_t n_points;    // N (point cloud size); windows W = N - 5
  uint64_t n_windows;
  uint32_t n_leaves;    // ceil(W / 8)
  int n_levels;         // node levels; the top level has <= 8 nodes
  uint32_t level_count[kMaxLevels];  // nodes per level
  uint32_t level_off[kMaxLevels];    // first uint2 of level L inside nodes[] (top level at 0)
  const uint2 *nodes;         // every level, top-down
  int smem_from;              // levels >= smem_from are staged in shared memory (n_levels: none)
  uint32_t smem_bytes;        // size of those levels = prefix of nodes[], multiple of 16
  const uint2 *leaves;        // [n_leaves][kLeafRec]: values, then {target position (pos >> 1, low
                              // 32 bits), contig*2 + strand (0 = '+'), ~0u = padding}
  const uint32_t *leaf_widx;  // [n_leaves*8] window index in the original cloud (parity hook only)
  float vmin, inv_span;       // Morton quantisation of the build: cell = (v - vmin) * inv_span
};

// one binary16 pair of a node record -> two floats
__device__ __forceinline__ float2 unpack_h2(uint32_t v) {
  return make_float2(__half2float(__ushort_as_half((unsigned short)(v & 0xFFFFu))),
                     __half2float(__ushort_as_half((unsigned short)(v >> 16))));
}

// order-preserving u32 image of a float (index extent and KD order) and its inverse
__device__ __forceinline__ uint32_t f2ord(float f) {
  const uint32_t u = __float_as_uint(f);
  return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__host__ __device__ __forceinline__ float ord2f(uint32_t o) {
  const uint32_t u = o ^ ((o >> 31) ? 0x80000000u : 0xFFFFFFFFu);
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  float f;
  memcpy(&f, &u, 4);
  return f;
#endif
}

// per-step packing of the 64-bit sort key: entry | bucket | target | query
struct KeyLayout {
  int qbits, tbits, bbits, ebits;
  __host__ __device__ int sh_t() const { return qbits; }
  __host__ __device__ int sh_b() const { return qbits + tbits; }
  __host__ __device__ int sh_e() const { return qbits + tbits + bbits; }
  __host__ __device__ int total() const { return qbits + tbits + bbits + ebits; }
  __host__ __device__ uint64_t pack(uint32_t e, uint32_t b, uint32_t t, uint32_t q) const {
    return ((uint64_t)e << sh_e()) | ((uint64_t)b << sh_b()) | ((uint64_t)t << sh_t()) | q;
  }
  __host__ __device__ uint32_t query(uint64_t k) const { return (uint32_t)(k & ((1ull << qbits) - 1)); }
  __host__ __device__ uint32_t target(uint64_t k) const { return (uint32_t)((k >> sh_t()) & ((1ull << tbits) - 1)); }
  __host__ __device__ uint32_t bucket(uint64_t k) const { return (uint32_t)((k >> sh_b()) & ((1ull << bbits) - 1)); }
  __host__ __device__ uint32_t entry(uint64_t k) const { return (uint32_t)(k >> sh_e()); }
  __host__ __device__ uint64_t seg(uint64_t k) const { return k >> sh_b(); }  // (entry, bucket)
};

// carried anchor (anchor of a surviving chain, re-injected next chunk: spatial_index.cc:303-322)
struct CarryAnchor {
  uint32_t target, query;
  float dist;
  uint32_t bucket;
};

// chain record kept per read slot between chunks (SignalAnchorChain minus the anchors)
struct ChainRec {
  float score;
  uint32_t contig, start, end, n_anchors, mapq, dir;
  uint32_t anchor_off;  // first anchor of this chain inside the slot's carry range
};

// per read-slot state carried between chunks + the last decision
struct SlotState {
  uint32_t num_events;   // query offset of the next chunk (sigmap.cc:666)
  uint32_t n_chains;
  uint32_t pool;         // which carry pool holds this slot's chains/anchors
  uint32_t owned0;       // 1: chain 0's anchors (and so ad/at/aq, q_first/q_last) are on this rank
  uint64_t chain_off;    // ChainRec index into pool_chain[pool]
  uint64_t carry_off;    // CarryAnchor index into pool_anchor[pool]
  uint32_t carry_n;
  uint32_t flags;        // bit0 query capped at 5000 hits; bit1 chain scratch overflow
  // decision inputs/outputs of the last GenerateChains (sigmap.cc:667-745)
  float s1, s2, sm, ad, at, aq;
  uint32_t cm, c0_contig, c0_start, c0_end, c0_dir, c0_mapq, q_first, q_last;
  uint32_t stop, mapped;
};

struct Counters {
  unsigned long long n_anchors;     // anchors written this step (hits + carried)
  unsigned long long n_hits;        // hits only
  unsigned long long n_queries;
  unsigned long long n_capped;
  unsigned long long n_events_raw;
  unsigned long long n_events_kept;
  unsigned long long n_linked;      // anchors with a gap-compatible predecessor (k_chain_prep)
  unsigned long long n_pending;     // of those, the ones k_chain_prep left to the DP kernels
  unsigned long long carry_anchor_used[2];
  unsigned long long carry_chain_used[2];
  unsigned long long sort_cursor;   // output position of the per-entry sort (k_seg_sort)
  unsigned long long n_cand;        // sharded: chain candidates this rank appended to its exchange list
  unsigned int n_segments;
  unsigned int work;                // dynamic work counter of the lean search kernel
  unsigned int work2;               // ... and of the general search kernel
  unsigned int n_overflow;          // queries the lean search kernel left to the general one
  unsigned int error;               // bit0 anchor overflow, bit1 carry overflow, bit2 chain scratch,
                                    // bit3 run table overflow, bit4 entry too dense for k_seg_sort,
                                    // bit5 candidate exchange list overflow
  unsigned int max_entry_anchors;   // most anchors any one (entry, part) received this step
  unsigned int dp_cursor;           // next segment of the chaining DP's work queue
  // The step runs without host round trips: what the host used to decide between kernels is
  // decided on the device.  A non-zero `abort` makes every later kernel of the step return at
  // once, so nothing is committed to the read slots and the host (which looks at the counters
  // once, at the end of the step) can redo the step with larger buffers or another sort path.
  unsigned int abort;               // kAbort* bits
  unsigned long long need_chain, need_anchor;  // carry-pool records the step's surviving chains need
};
constexpr unsigned int kAbortAnchors = 1u;  // more anchors than the step's buffers hold
constexpr unsigned int kAbortSort = 2u;     // the chosen sort path cannot take this step (run tables, dense part)
constexpr unsigned int kAbortQueries = 4u;  // more queries than the order buffers hold
constexpr unsigned int kAbortPool = 8u;     // carry pools too small for the surviving chains

// The index build sets the shift that puts every g of the index below kCoarseBins (k_seg_sort).
constexpr int kCoarseBins = 256;

// Part of an entry that linear coordinate g = bucket_base[bucket] + target belongs to
// (k_sort.cuh, k_part_sort).  Any function that is monotone in g gives contiguous parts; float
// rounding only moves the boundaries by a few hundred positions, identically for every producer.
__host__ __device__ __forceinline__ uint32_t part_of(uint64_t g, float inv_span, uint32_t n_parts) {
  const uint32_t p = (uint32_t)((float)g * inv_span);
  return p < n_parts ? p : n_parts - 1u;
}

// where one flush of the search kernel (or the carry injection) wrote hits of one entry
struct RunRec {
  uint32_t start, count;
};

}  // namespace sb
#endif
