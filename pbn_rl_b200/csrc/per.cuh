// Prioritised experience replay on the device: sum / min priority trees over the replay ring's slots,
// proportional stratified sampling and importance weights (contract: include/pbn_b200.h, "Prioritised replay").
//
// The reference's PER (SURVEY.md section 2 row 14, data_structures.py) is a numpy segment tree updated one leaf at a
// time.  Here the whole binary tree is stored as a heap in one caller-owned float array (layout in the header), so
// every binary node the contract defines is materialised and can be compared bit for bit:
//   - push rebuilds the dirty leaf ranges tile by tile in shared memory (one CTA per tile of 2^kPerTileLog2 leaves)
//     and the last CTA to finish recomputes the levels above the tile roots;
//   - update (B <= kPerUpdateOneCta) is one CTA: last-wins through a per-slot owner word, leaves, then the dirty
//     ancestors level by level behind __syncthreads; larger batches claim / write with the whole grid and rebuild
//     the tree with the push kernel;
//   - sample is a warp per sample: the warp loads the 32 descendants five binary levels below the current node,
//     rebuilds the four levels in between with shuffles (the same fp32 adds, and fp32 addition is commutative, so
//     the values equal the stored nodes) and takes five binary decisions from registers: ceil(log2 L / 5) dependent
//     loads instead of log2 L.
#pragma once
#include "pbn_common.cuh"

namespace pbn {

constexpr int kPerTileLog2 = 11;        // leaves per push / rebuild CTA (shared memory: 4 * 2^11 floats = 32 KB)
constexpr int kPerRebuildThreads = 512;
constexpr int kPerUpdateThreads = 1024;
constexpr int64_t kPerUpdateOneCta = 4096;   // largest batch of the single-CTA update

struct PerView {
  float* sum;                 // heap: node k at sum[k], leaves at sum[L + slot]
  float* mn;                  // the min tree, same indexing
  int* owner;                 // [L] last batch position that wrote a slot (-1 between calls)
  unsigned int* ticket;       // completion ticket of the rebuild kernel (0 between calls)
  float* max_p;
  int64_t L, capacity;
  int D;                      // log2 L
  float alpha;
};

// slot ranges [a0, b0) and [a1, b1) whose leaves a push sets (empty ranges: a == b); tiles of the grid: blocks
// [0, n0) take tiles t0.., blocks [n0, grid) take tiles t1..
struct PerRanges {
  int64_t a0, b0, a1, b1;
  int64_t t0, n0, t1;
  int lt;                     // log2 of the tile size (min(kPerTileLog2, D))
  int fill;                   // 0: rebuild only (the ranges still bound the top pass)
};

__device__ __forceinline__ float per_clamp(float td, float eps) {
  return fminf(__fadd_rn(fmaxf(fabsf(td), 0.0f), eps), 1e30f);
}

__global__ void __launch_bounds__(256) per_init_kernel(PerView v) {
  const int64_t nth = (int64_t)gridDim.x * blockDim.x, tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t i = tid; i < 2 * v.L; i += nth) {
    v.sum[i] = 0.0f;
    v.mn[i] = __int_as_float(0x7f800000);
  }
  for (int64_t i = tid; i < v.L; i += nth) v.owner[i] = -1;
  if (tid == 0) {
    *v.ticket = 0u;
    *v.max_p = 1.0f;
  }
}

// Leaves of the pushed ranges <- powf(max_p, alpha) and every ancestor of them rebuilt (fill = 0: no leaf is set,
// the ancestors of the ranges are rebuilt from the stored leaves).  reset_index[0..reset_n): owner words to clear
// (the multi-CTA update path).
__global__ void __launch_bounds__(kPerRebuildThreads) per_rebuild_kernel(PerView v, PerRanges r,
                                                                         const int64_t* __restrict__ reset_index,
                                                                         int64_t reset_n) {
  __shared__ float hs[2 << kPerTileLog2], hm[2 << kPerTileLog2];
  __shared__ bool last;
  const int te = 1 << r.lt;
  const int64_t tile = blockIdx.x < r.n0 ? r.t0 + blockIdx.x : r.t1 + (blockIdx.x - r.n0);
  const int64_t base = tile << r.lt;
  const float val = r.fill ? powf(*v.max_p, v.alpha) : 0.0f;
  for (int i = threadIdx.x; i < te; i += blockDim.x) {
    const int64_t slot = base + i;
    const bool in = r.fill && ((slot >= r.a0 && slot < r.b0) || (slot >= r.a1 && slot < r.b1));
    float s, m;
    if (in) {
      s = m = val;
      v.sum[v.L + slot] = val;
      v.mn[v.L + slot] = val;
    } else {
      s = v.sum[v.L + slot];
      m = v.mn[v.L + slot];
    }
    hs[te + i] = s;
    hm[te + i] = m;
  }
  const int64_t root = (v.L >> r.lt) + tile;   // heap index of the tile's root
  for (int n = te >> 1, d = r.lt - 1; n >= 1; n >>= 1, --d) {
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int k = n + i;
      const float s = __fadd_rn(hs[2 * k], hs[2 * k + 1]), m = fminf(hm[2 * k], hm[2 * k + 1]);
      hs[k] = s;
      hm[k] = m;
      const int64_t g = (root << d) + i;   // n = 2^d nodes at depth d below the tile root
      v.sum[g] = s;
      v.mn[g] = m;
    }
  }
  if (reset_index) {
    const int64_t nth = (int64_t)gridDim.x * blockDim.x, tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t b = tid; b < reset_n; b += nth) {
      const int64_t s = reset_index[b];
      if (s >= 0 && s < v.capacity) v.owner[s] = -1;
    }
  }
  // the last CTA to finish rebuilds the levels above the tile roots
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicAdd(v.ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  const int64_t lo[2] = {r.a0, r.a1}, hi[2] = {r.b0, r.b1};
  for (int k = r.lt + 1; k <= v.D; ++k) {
    for (int q = 0; q < 2; ++q) {
      if (hi[q] <= lo[q]) continue;
      const int64_t n0 = (v.L + lo[q]) >> k, n1 = (v.L + hi[q] - 1) >> k;
      for (int64_t g = n0 + threadIdx.x; g <= n1; g += blockDim.x) {
        v.sum[g] = __fadd_rn(__ldcg(v.sum + 2 * g), __ldcg(v.sum + 2 * g + 1));
        v.mn[g] = fminf(__ldcg(v.mn + 2 * g), __ldcg(v.mn + 2 * g + 1));
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) *v.ticket = 0u;
}

// max_p <- max(max_p, raw of every valid batch entry): raw > 0 and finite, so the bit patterns order like the values
__device__ __forceinline__ void per_fold_max(PerView v, float raw) {
  for (int o = 16; o; o >>= 1) raw = fmaxf(raw, __shfl_xor_sync(0xffffffffu, raw, o));
  if ((threadIdx.x & 31) == 0 && raw > 0.0f) atomicMax(reinterpret_cast<int*>(v.max_p), __float_as_int(raw));
}

// the batch entry that owns its slot (the last occurrence in batch order) writes the leaf; returns its raw priority
// (0 for an out-of-range index) for the max_p fold
__device__ __forceinline__ float per_write_leaf(PerView v, const int64_t* index, const float* td, int64_t b, float eps) {
  const int64_t s = index[b];
  if (s < 0 || s >= v.capacity) return 0.0f;
  const float raw = per_clamp(td[b], eps);
  if (__ldcg(v.owner + s) == (int)b) {
    const float p = powf(raw, v.alpha);
    v.sum[v.L + s] = p;
    v.mn[v.L + s] = p;
  }
  return raw;
}

// The whole update of a batch of at most kPerUpdateOneCta entries in one CTA.
__global__ void __launch_bounds__(kPerUpdateThreads) per_update_cta_kernel(PerView v, const int64_t* __restrict__ index,
                                                                           const float* __restrict__ td, int B,
                                                                           float eps) {
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const int64_t s = index[b];
    if (s >= 0 && s < v.capacity) atomicMax(v.owner + s, b);
  }
  __syncthreads();
  float raw = 0.0f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) raw = fmaxf(raw, per_write_leaf(v, index, td, b, eps));
  per_fold_max(v, raw);
  __syncthreads();
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const int64_t s = index[b];
    if (s >= 0 && s < v.capacity) v.owner[s] = -1;
  }
  for (int k = 1; k <= v.D; ++k) {
    __syncthreads();
    const int64_t nodes = v.L >> k;
    if (nodes <= blockDim.x) {   // narrow level: every node once, no duplicates
      for (int64_t g = nodes + threadIdx.x; g < 2 * nodes; g += blockDim.x) {
        v.sum[g] = __fadd_rn(__ldcg(v.sum + 2 * g), __ldcg(v.sum + 2 * g + 1));
        v.mn[g] = fminf(__ldcg(v.mn + 2 * g), __ldcg(v.mn + 2 * g + 1));
      }
    } else {                     // wide level: the ancestor of each entry (duplicates write the same values)
      for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const int64_t s = index[b];
        if (s < 0 || s >= v.capacity) continue;
        const int64_t g = (v.L + s) >> k;
        v.sum[g] = __fadd_rn(__ldcg(v.sum + 2 * g), __ldcg(v.sum + 2 * g + 1));
        v.mn[g] = fminf(__ldcg(v.mn + 2 * g), __ldcg(v.mn + 2 * g + 1));
      }
    }
  }
}

// Larger batches, first pass: claim the slots (the rebuild kernel clears the claims afterwards).
__global__ void __launch_bounds__(256) per_update_claim_kernel(PerView v, const int64_t* __restrict__ index, int64_t B) {
  const int64_t nth = (int64_t)gridDim.x * blockDim.x, tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t b = tid; b < B; b += nth) {
    const int64_t s = index[b];
    if (s >= 0 && s < v.capacity) atomicMax(v.owner + s, (int)b);
  }
}

// Larger batches, second pass: the owners write their leaves.
__global__ void __launch_bounds__(256) per_update_write_kernel(PerView v, const int64_t* __restrict__ index,
                                                               const float* __restrict__ td, int64_t B, float eps) {
  const int64_t nth = (int64_t)gridDim.x * blockDim.x, tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float raw = 0.0f;
  for (int64_t b = tid; b < B; b += nth) raw = fmaxf(raw, per_write_leaf(v, index, td, b, eps));
  per_fold_max(v, raw);
}

// Stratified proportional sampling, one warp per sample (see the top of this file).
__global__ void __launch_bounds__(256) per_sample_kernel(PerView v, const float* __restrict__ u, int64_t B, float beta,
                                                         int64_t* __restrict__ index, float* __restrict__ weight) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const float total = __ldg(v.sum + 1), pmin = __ldg(v.mn + 1);
  const float seg = __fdiv_rn(total, (float)B);
  for (int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < B; b += nw) {
    float mass = __fadd_rn(__fmul_rn(u[b], seg), __fmul_rn((float)b, seg));
    int64_t g = 1;
    for (int rem = v.D; rem > 0;) {
      const int w = rem < 5 ? rem : 5;
      const int64_t base = g << w;
      float t[5];
      t[0] = lane < (1 << w) ? __ldg(v.sum + base + lane) : 0.0f;
#pragma unroll
      for (int j = 1; j < 5; ++j) t[j] = __fadd_rn(t[j - 1], __shfl_xor_sync(0xffffffffu, t[j - 1], 1 << (j - 1)));
      int cur = 0;   // index of the current node among the 2^(w-j-1) nodes of its sub-level
#pragma unroll
      for (int j = 4; j >= 0; --j) {
        if (j >= w) continue;
        const float left = __shfl_sync(0xffffffffu, t[j], (2 * cur) << j);
        const float right = __shfl_sync(0xffffffffu, t[j], (2 * cur + 1) << j);
        if (left > mass || right == 0.0f) {
          cur = 2 * cur;
        } else {
          mass = __fsub_rn(mass, left);
          cur = 2 * cur + 1;
        }
      }
      g = base + cur;
      rem -= w;
    }
    if (lane == 0) {
      const int64_t s = g - v.L;
      index[b] = s;
      weight[b] = powf(__fdiv_rn(pmin, __ldg(v.sum + g)), beta);
    }
  }
}

}  // namespace pbn
