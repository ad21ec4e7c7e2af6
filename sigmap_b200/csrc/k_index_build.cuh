// k_index_build.cuh -- build kernels of the flat device index (k_index.cuh): the aligned KD
// order of the windows, the leaf records and the node levels (layout: IndexView, sb_device.cuh).
// Launched by build_index_core in sb_index.cu.
#ifndef SB_K_INDEX_BUILD_CUH
#define SB_K_INDEX_BUILD_CUH

#include <cuda_fp16.h>

#include "sb_device.cuh"

namespace sb {

// ---- aligned KD order (the default point order).  The pointer-free hierarchy puts node k of level
// l over the points [k * 8^(l+1), (k+1) * 8^(l+1)) of the order, so any order works; what the search
// pays for is how tight those groups are.  Morton order cuts space at fixed midpoints and a group of
// 8^k consecutive codes can straddle a large cell boundary; here every power-of-two-aligned group
// is a KD cell instead: for s = 2^k >= W down to 16, every aligned segment of s positions is sorted
// along the dimension in which its points spread most, so its lower half (the next level's left
// segment) is a half-space cut of it.  Measured on config 2 (tools/emulate_kd.py): 334 box tests per
// query instead of 679, 28.6 leaves instead of 31.7.
//   k_kd_extent  per-segment min / max of the six coordinates (order-preserving u32 images)
//   k_kd_keys    key = segment << 32 | image of the coordinate along the segment's widest dimension
//   (one stable radix sort of (key, window) per level in between)
constexpr int kKdThreads = 256;

// idx == nullptr: the identity order (first level)
__global__ void __launch_bounds__(kKdThreads)
k_kd_extent(const float *__restrict__ val, const uint32_t *__restrict__ idx, const uint32_t *__restrict__ wsrc,
            uint64_t W, int log2s, uint32_t *__restrict__ ext_min, uint32_t *__restrict__ ext_max) {
  __shared__ uint32_t s_red[kKdThreads / 32][2 * kDim];
  const uint64_t i = (uint64_t)blockIdx.x * kKdThreads + threadIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t mn[kDim], mx[kDim];
#pragma unroll
  for (int d = 0; d < kDim; ++d) {
    mn[d] = 0xFFFFFFFFu;
    mx[d] = 0u;
  }
  if (i < W) {
    const uint32_t w = idx ? idx[i] : (uint32_t)i;
    const uint64_t v0 = wsrc ? (uint64_t)wsrc[w] : (uint64_t)w;
#pragma unroll
    for (int d = 0; d < kDim; ++d) mn[d] = mx[d] = f2ord(val[v0 + d]);
  }
  // lanes that share a segment: the whole warp (log2s >= 5) or each half of it (log2s == 4)
  const unsigned m = log2s >= 5 ? 0xFFFFFFFFu : (lane < 16 ? 0x0000FFFFu : 0xFFFF0000u);
#pragma unroll
  for (int d = 0; d < kDim; ++d) {
    mn[d] = __reduce_min_sync(m, mn[d]);
    mx[d] = __reduce_max_sync(m, mx[d]);
  }
  if (log2s >= 8) {  // the whole block lies in one segment: one set of atomics per block
    if (lane == 0) {
#pragma unroll
      for (int d = 0; d < kDim; ++d) {
        s_red[wid][d] = mn[d];
        s_red[wid][kDim + d] = mx[d];
      }
    }
    __syncthreads();
    if (threadIdx.x < 2 * kDim) {
      const bool is_max = threadIdx.x >= kDim;
      uint32_t r = s_red[0][threadIdx.x];
      for (int w = 1; w < kKdThreads / 32; ++w) r = is_max ? max(r, s_red[w][threadIdx.x]) : min(r, s_red[w][threadIdx.x]);
      const uint64_t seg = ((uint64_t)blockIdx.x * kKdThreads) >> log2s;
      if ((uint64_t)blockIdx.x * kKdThreads < W) {
        if (is_max) atomicMax(&ext_max[seg * kDim + (threadIdx.x - kDim)], r);
        else atomicMin(&ext_min[seg * kDim + threadIdx.x], r);
      }
    }
  } else if (i < W && (lane == 0 || (log2s == 4 && lane == 16))) {
    const uint64_t seg = i >> log2s;
#pragma unroll
    for (int d = 0; d < kDim; ++d) {
      atomicMin(&ext_min[seg * kDim + d], mn[d]);
      atomicMax(&ext_max[seg * kDim + d], mx[d]);
    }
  }
}

__global__ void __launch_bounds__(kKdThreads)
k_kd_keys(const float *__restrict__ val, const uint32_t *__restrict__ idx, const uint32_t *__restrict__ wsrc,
          uint64_t W, int log2s, const uint32_t *__restrict__ ext_min, const uint32_t *__restrict__ ext_max,
          uint64_t *__restrict__ key, uint32_t *__restrict__ idx_out) {
  const uint64_t i = (uint64_t)blockIdx.x * kKdThreads + threadIdx.x;
  if (i >= W) return;
  const uint64_t seg = i >> log2s;
  int dim = 0;
  float widest = -1.0f;
#pragma unroll
  for (int d = 0; d < kDim; ++d) {
    const float e = ord2f(ext_max[seg * kDim + d]) - ord2f(ext_min[seg * kDim + d]);
    if (e > widest) {  // ties: the lowest dimension
      widest = e;
      dim = d;
    }
  }
  const uint32_t w = idx ? idx[i] : (uint32_t)i;
  const uint64_t v0 = wsrc ? (uint64_t)wsrc[w] : (uint64_t)w;
  key[i] = (seg << 32) | (uint64_t)f2ord(val[v0 + dim]);
  if (!idx) idx_out[i] = w;
}

// sorted rank i -> leaf records; one thread per slot of the padded leaf array.  order == nullptr:
// rank i is window i (an index of one leaf)
__global__ void k_build_leaves(const float *__restrict__ val, const uint64_t *__restrict__ pos,
                               const uint32_t *__restrict__ order, uint64_t n_windows,
                               uint32_t n_leaves, uint2 *__restrict__ leaves,
                               uint32_t *__restrict__ leaf_widx,
                               const uint32_t *__restrict__ wsrc, const uint32_t *__restrict__ worig) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (uint64_t)n_leaves * kLeaf) return;
  const uint32_t leaf = (uint32_t)(i / kLeaf), sub = (uint32_t)(i % kLeaf);
  uint2 *rec = leaves + (size_t)leaf * kLeafRec + sub;
  float2 *v = reinterpret_cast<float2 *>(rec);
  if (i < n_windows) {
    const uint32_t w = order ? order[i] : (uint32_t)i;
    const uint64_t v0 = wsrc ? (uint64_t)wsrc[w] : (uint64_t)w;
#pragma unroll
    for (int k = 0; k < 3; ++k) v[k * kLeaf] = make_float2(val[v0 + 2 * k], val[v0 + 2 * k + 1]);
    const uint64_t P = pos[w];
    // target = pos >> 1 (spatial_index.cc:380-381); bucket = contig*2 + strand
    rec[3 * kLeaf] = make_uint2((uint32_t)(P >> 1), (uint32_t)((P >> 33) << 1) | (uint32_t)(P & 1));
    leaf_widx[i] = worig ? worig[w] : w;
  } else {
#pragma unroll
    for (int k = 0; k < 3; ++k) v[k * kLeaf] = make_float2(kPadValue, kPadValue);
    rec[3 * kLeaf] = make_uint2(0u, 0xFFFFFFFFu);
    leaf_widx[i] = 0xFFFFFFFFu;
  }
}

// box [lo, hi] -> twelve binary16 numbers, lo rounded down and hi rounded up, so the stored box
// always contains the fp32 one (values beyond the binary16 range become +-inf: never pruned);
// stored as child `j` of node record `rec`.  A padding child is the empty box (+inf, -inf).
__device__ __forceinline__ uint32_t pack_h2(__half a, __half b) {
  return (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16);
}
__device__ __forceinline__ void store_child_box(uint2 *rec, int j, const float *lo, const float *hi, bool real) {
  __half l[kDim], h[kDim];
#pragma unroll
  for (int d = 0; d < kDim; ++d) {
    if (real) {
      l[d] = __float2half_rd(lo[d]);
      h[d] = __float2half_ru(hi[d]);
    } else {
      l[d] = __ushort_as_half((unsigned short)0x7C00);  // +inf
      h[d] = __ushort_as_half((unsigned short)0xFC00);  // -inf
    }
  }
  rec[j] = make_uint2(pack_h2(l[0], l[1]), pack_h2(l[2], l[3]));
  rec[kFan + j] = make_uint2(pack_h2(l[4], l[5]), pack_h2(h[0], h[1]));
  rec[2 * kFan + j] = make_uint2(pack_h2(h[2], h[3]), pack_h2(h[4], h[5]));
}
// child `j` of a node record -> lo[6], hi[6]
__device__ __forceinline__ void load_child_box(const uint2 *rec, int j, float *lo, float *hi) {
  const uint2 a = rec[j], b = rec[kFan + j], c = rec[2 * kFan + j];
  const float2 l01 = unpack_h2(a.x), l23 = unpack_h2(a.y), l45 = unpack_h2(b.x);
  const float2 h01 = unpack_h2(b.y), h23 = unpack_h2(c.x), h45 = unpack_h2(c.y);
  lo[0] = l01.x; lo[1] = l01.y; lo[2] = l23.x; lo[3] = l23.y; lo[4] = l45.x; lo[5] = l45.y;
  hi[0] = h01.x; hi[1] = h01.y; hi[2] = h23.x; hi[3] = h23.y; hi[4] = h45.x; hi[5] = h45.y;
}

// level-0 nodes: thread (n, j) boxes leaf 8n + j
__global__ void k_nodes_level0(const uint2 *__restrict__ leaves, uint32_t n_leaves, uint32_t n_nodes,
                               uint2 *__restrict__ nodes) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_nodes * kFan) return;
  const uint32_t n = t / kFan, j = t % kFan, leaf = t;
  float lo[kDim], hi[kDim];
#pragma unroll
  for (int d = 0; d < kDim; ++d) {
    lo[d] = 3.0e38f;
    hi[d] = -3.0e38f;
  }
  bool real = false;
  if (leaf < n_leaves) {
    const uint2 *rec = leaves + (size_t)leaf * kLeafRec;
    for (int p = 0; p < kLeaf; ++p) {
      if (rec[3 * kLeaf + p].y == 0xFFFFFFFFu) continue;
      real = true;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const uint2 raw = rec[k * kLeaf + p];
        const float2 v = make_float2(__uint_as_float(raw.x), __uint_as_float(raw.y));
        lo[2 * k] = fminf(lo[2 * k], v.x);
        hi[2 * k] = fmaxf(hi[2 * k], v.x);
        lo[2 * k + 1] = fminf(lo[2 * k + 1], v.y);
        hi[2 * k + 1] = fmaxf(hi[2 * k + 1], v.y);
      }
    }
  }
  store_child_box(nodes + (size_t)n * 3 * kFan, (int)j, lo, hi, real);
}

// level l+1 from level l: thread (n, j) boxes child node 8n + j of the level below
__global__ void k_nodes_up(const uint2 *__restrict__ child, uint32_t n_child, uint32_t n_nodes,
                           uint2 *__restrict__ nodes) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_nodes * kFan) return;
  const uint32_t n = t / kFan, j = t % kFan, m = t;
  float lo[kDim], hi[kDim];
#pragma unroll
  for (int d = 0; d < kDim; ++d) {
    lo[d] = 3.0e38f;
    hi[d] = -3.0e38f;
  }
  bool real = false;
  if (m < n_child) {
    const uint2 *rec = child + (size_t)m * 3 * kFan;
    for (int p = 0; p < kFan; ++p) {
      float cl[kDim], ch[kDim];
      load_child_box(rec, p, cl, ch);
      if (cl[0] > ch[0]) continue;  // padding child (empty box)
      real = true;
#pragma unroll
      for (int d = 0; d < kDim; ++d) {
        lo[d] = fminf(lo[d], cl[d]);
        hi[d] = fmaxf(hi[d], ch[d]);
      }
    }
  }
  store_child_box(nodes + (size_t)n * 3 * kFan, (int)j, lo, hi, real);
}

}  // namespace sb
#endif
