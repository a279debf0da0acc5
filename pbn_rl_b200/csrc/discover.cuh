// Attractor discovery / steady-state statistics support (SURVEY.md 8f-3): a visit-count hash table in
// HBM.  Massive perturbation-free rollouts (pbn_step) end in the network's attractors; counting the
// distinct end states on the device replaces the reference's per-instance bookkeeping
// (env.all_attractors growing during training, bdq_model/__init__.py:182-184; compute_ssd_hist's
// state histogram, train_pbn_28.py:257).  Open addressing, linear probing, capacity a power of two.
#pragma once
#include "pbn_common.cuh"

namespace pbn {

// Key of a state in the tags[] column: never 0 (empty slot) and never 1 (kTagBusy).
//   W == 1, N <= 63: tag = 2*state + 1  -- injective: distinct states never share a slot.
//   otherwise      : a 64-bit splitmix64 fingerprint; a tag match is confirmed by comparing the state words in
//                    slot_state (the claimer publishes them BEFORE the tag becomes visible), so distinct states
//                    with equal fingerprints occupy different slots instead of being merged.
constexpr unsigned long long kTagBusy = 1ull;

template <int W>
__device__ __forceinline__ uint64_t state_tag(const uint64_t (&s)[W], bool injective) {
  if (W == 1 && injective) return (s[0] << 1) | 1ull;
  uint64_t h = mix64(s[0] + 0x9E3779B97F4A7C15ull);
  if (W == 2) h = mix64(h ^ (s[1] + 0xD1B54A32D192ED03ull));
  return h < 2ull ? h + 2ull : h;
}

constexpr int kMaxProbe = 4096;

template <int W>
__device__ __forceinline__ bool slot_holds(const uint64_t* __restrict__ slot_state, uint64_t slot, const uint64_t (&s)[W]) {
  bool same = true;
#pragma unroll
  for (int w = 0; w < W; ++w) same = same && reinterpret_cast<const volatile uint64_t*>(slot_state)[slot * W + w] == s[w];
  return same;
}

// Insert-or-find in the open-addressing table: returns the slot (or -1 if no slot within kMaxProbe probes);
// fresh = this call claimed the slot (exactly one caller per distinct state sees fresh = true).
// Claim protocol: CAS 0 -> kTagBusy, write the state words, fence, store the tag.  A prober that meets kTagBusy
// waits (bounded) for the tag: the claimer is always a running thread that needs nothing from the prober.
template <int W>
__device__ __forceinline__ int64_t hash_insert(const uint64_t (&s)[W], unsigned long long* __restrict__ tags,
                                               uint64_t* __restrict__ slot_state, uint64_t cap_mask, bool injective,
                                               bool& fresh) {
  const uint64_t tag = state_tag<W>(s, injective);
  uint64_t slot = mix64(tag) & cap_mask;
  fresh = false;
  for (int probe = 0; probe < kMaxProbe; ++probe, slot = (slot + 1) & cap_mask) {
    unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(&tags[slot]);
    if (cur == 0ull) {
      cur = atomicCAS(&tags[slot], 0ull, kTagBusy);
      if (cur == 0ull) {
#pragma unroll
        for (int w = 0; w < W; ++w) slot_state[slot * W + w] = s[w];
        __threadfence();
        atomicExch(&tags[slot], (unsigned long long)tag);
        fresh = true;
        return (int64_t)slot;
      }
    }
    for (int spin = 0; cur == kTagBusy && spin < (1 << 16); ++spin) {
      __nanosleep(20);
      cur = *reinterpret_cast<volatile unsigned long long*>(&tags[slot]);
    }
    if (cur == tag && ((W == 1 && injective) || slot_holds<W>(slot_state, slot, s))) return (int64_t)slot;
  }
  return -1;
}

template <int W>
__device__ __forceinline__ int64_t hash_find(const uint64_t (&s)[W], const unsigned long long* __restrict__ tags,
                                             const uint64_t* __restrict__ slot_state, uint64_t cap_mask, bool injective) {
  const uint64_t tag = state_tag<W>(s, injective);
  uint64_t slot = mix64(tag) & cap_mask;
  for (int probe = 0; probe < kMaxProbe; ++probe, slot = (slot + 1) & cap_mask) {
    const unsigned long long cur = tags[slot];
    if (cur == tag && ((W == 1 && injective) || slot_holds<W>(slot_state, slot, s))) return (int64_t)slot;
    if (cur == 0ull) return -1;
  }
  return -1;
}

// counts[slot(state[e])] += 1 for every instance with mask[e] != 0 (all if mask == nullptr).
// tags[cap] (0 = empty), slot_state[cap*W], counts[cap]; *overflow counts states that found no slot
// within kMaxProbe probes (table too full).
template <int W>
__global__ void __launch_bounds__(256) visit_count_kernel(const uint64_t* __restrict__ state, const uint8_t* __restrict__ mask,
                                                         int64_t n_envs, unsigned long long* __restrict__ tags,
                                                         uint64_t* __restrict__ slot_state,
                                                         unsigned long long* __restrict__ counts, uint64_t cap_mask,
                                                         bool injective, unsigned int* __restrict__ overflow) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_envs; e += (int64_t)gridDim.x * blockDim.x) {
    if (mask != nullptr && mask[e] == 0) continue;
    uint64_t s[W];
#pragma unroll
    for (int w = 0; w < W; ++w) s[w] = state[e * W + w];
    bool fresh;
    const int64_t slot = hash_insert<W>(s, tags, slot_state, cap_mask, injective, fresh);
    if (slot >= 0) atomicAdd(&counts[slot], 1ull); else atomicAdd(overflow, 1u);
  }
}

// Value (0 or 1) of predictor function f in state s: the narrow 64-bit truth table or a wide one.  Shared by the
// successor descriptor below and the exact backup of control.cuh, so both see the same predictor values.
template <int W>
__device__ __forceinline__ uint64_t eval_func(const NetParams& n, int f, const uint64_t (&s)[W]) {
  const FuncDesc d = n.funcs[f];
  uint64_t v;
  if (d.in47 == kWideMarker) {
    v = eval_wide<W>(n, d.lut_lo, s);
  } else {
    uint32_t idx = 0;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const uint32_t in = ((j < 4 ? d.in03 >> (8 * j) : d.in47 >> (8 * (j - 4))) & 0xFFu);
      idx |= (uint32_t)((s[W == 1 ? 0 : (in >> 6)] >> (in & 63u)) & 1ull) << j;
    }
    const uint64_t lut = ((uint64_t)d.lut_hi << 32) | d.lut_lo;   // replicated over unused inputs
    v = (lut >> idx) & 1ull;
  }
  return v;
}

// (can1, can0) of one state: which genes some predictor can set to 1 / to 0 in one perturbation-free update.
template <int W>
__device__ __forceinline__ void successor_descriptor(const NetParams& n, const uint64_t (&s)[W], uint64_t (&c1)[W],
                                                     uint64_t (&c0)[W]) {
#pragma unroll
  for (int w = 0; w < W; ++w) { c1[w] = 0; c0[w] = 0; }
  for (int g = 0; g < n.n_genes; ++g) {
    for (int f = n.func_offset[g]; f < n.func_offset[g + 1]; ++f) {
      const uint64_t v = eval_func<W>(n, f, s);
      c1[g >> 6] |= v << (g & 63);
      c0[g >> 6] |= (v ^ 1ull) << (g & 63);
    }
  }
}

// Per state of a list: the successor descriptor of the state-transition graph (graph.genSTG(),
// print_graph.py:15-21): successors = {fixed bits} x {0,1}^(genes that can do both).
template <int W>
__global__ void __launch_bounds__(256) successor_sets_kernel(const __grid_constant__ NetParams n,
                                                            const uint64_t* __restrict__ state, int64_t n_states,
                                                            uint64_t* __restrict__ can1, uint64_t* __restrict__ can0) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_states; e += (int64_t)gridDim.x * blockDim.x) {
    uint64_t s[W], c1[W], c0[W];
#pragma unroll
    for (int w = 0; w < W; ++w) s[w] = state[e * W + w];
    successor_descriptor<W>(n, s, c1, c0);
#pragma unroll
    for (int w = 0; w < W; ++w) { can1[e * W + w] = c1[w]; can0[e * W + w] = c0[w]; }
  }
}

// ---- forward closure and backward reachability on the device (exact attractors of large networks) ----
// The closure of a candidate state is kept as a list (discovery order) plus the hash table above, whose
// counts[] column stores list index + 1.  One CTA handles one list entry: thread 0 derives the successor
// descriptor, all threads enumerate the 2^free successors.
constexpr int kClosureMaxFree = 20;
enum { kClosureOk = 0, kClosureTooManyFree = 1, kClosureListFull = 2, kClosureTableFull = 3 };

template <int W>
struct ClosureShared {
  uint64_t fixed[W];
  int pos[kClosureMaxFree];
  int nfree;
  int abort;
};

template <int W>
__device__ __forceinline__ void closure_prepare(const NetParams& n, const uint64_t* __restrict__ list, int64_t i,
                                                ClosureShared<W>& sh, const int* status = nullptr) {
  if (threadIdx.x == 0) {
    sh.abort = status != nullptr ? *reinterpret_cast<const volatile int*>(status) : 0;
    uint64_t s[W], c1[W], c0[W];
#pragma unroll
    for (int w = 0; w < W; ++w) s[w] = list[i * W + w];
    successor_descriptor<W>(n, s, c1, c0);
    int nf = 0;
#pragma unroll
    for (int w = 0; w < W; ++w) {
      uint64_t fr = c1[w] & c0[w];
      sh.fixed[w] = c1[w] & ~fr;
      while (fr) {
        const int b = __ffsll((long long)fr) - 1;
        if (nf < kClosureMaxFree) sh.pos[nf] = 64 * w + b;
        ++nf;
        fr &= fr - 1;
      }
    }
    sh.nfree = nf;
  }
  __syncthreads();
}

template <int W>
__device__ __forceinline__ void closure_successor(const ClosureShared<W>& sh, uint32_t j, uint64_t (&t)[W]) {
#pragma unroll
  for (int w = 0; w < W; ++w) t[w] = sh.fixed[w];
  for (int b = 0; b < sh.nfree; ++b)
    if ((j >> b) & 1u) t[sh.pos[b] >> 6] |= 1ull << (sh.pos[b] & 63);
}

// Expand list[begin, end): every successor not yet in the table is appended to the list.
template <int W>
__global__ void __launch_bounds__(128) closure_expand_kernel(const __grid_constant__ NetParams n, uint64_t* __restrict__ list,
                                                            int64_t begin, int64_t end, int64_t list_cap,
                                                            unsigned long long* __restrict__ list_count,
                                                            unsigned long long* __restrict__ tags,
                                                            uint64_t* __restrict__ slot_state,
                                                            unsigned long long* __restrict__ slot_index, uint64_t cap_mask,
                                                            int max_free, int* __restrict__ status) {
  __shared__ ClosureShared<W> sh;
  for (int64_t i = begin + blockIdx.x; i < end; i += gridDim.x) {
    closure_prepare<W>(n, list, i, sh, status);
    if (sh.abort != 0) break;   // another CTA already ran out of room: the search has failed, stop early
    if (sh.nfree > max_free || sh.nfree > kClosureMaxFree) {
      if (threadIdx.x == 0) atomicMax(status, (int)kClosureTooManyFree);
    } else {
      const uint32_t total = 1u << sh.nfree;
      for (uint32_t j = threadIdx.x; j < total; j += blockDim.x) {
        uint64_t t[W];
        closure_successor<W>(sh, j, t);
        bool fresh;
        const int64_t slot = hash_insert<W>(t, tags, slot_state, cap_mask, W == 1 && n.n_genes <= 63, fresh);
        if (slot < 0) {
          atomicMax(status, (int)kClosureTableFull);
        } else if (fresh) {
          const unsigned long long k = atomicAdd(list_count, 1ull);
          if ((int64_t)k < list_cap) {
#pragma unroll
            for (int w = 0; w < W; ++w) list[k * W + w] = t[w];
            slot_index[slot] = k + 1ull;
          } else {
            atomicMax(status, (int)kClosureListFull);
          }
        }
      }
    }
    __syncthreads();
  }
}

// One sweep of backward reachability inside the closed set: an entry whose flag is 0 gets flag 1 if one of its
// successors has flag 1.  Repeated by the host until *changed stays 0; flags[i] = 1 then means "list[i] reaches
// the seed".
template <int W>
__global__ void __launch_bounds__(128) closure_reach_kernel(const __grid_constant__ NetParams n, const uint64_t* __restrict__ list,
                                                           int64_t count, uint8_t* __restrict__ flags,
                                                           const unsigned long long* __restrict__ tags,
                                                           const uint64_t* __restrict__ slot_state,
                                                           const unsigned long long* __restrict__ slot_index,
                                                           uint64_t cap_mask, int* __restrict__ changed) {
  __shared__ ClosureShared<W> sh;
  const bool injective = W == 1 && n.n_genes <= 63;
  for (int64_t i = blockIdx.x; i < count; i += gridDim.x) {
    if (flags[i] != 0) continue;      // uniform across the CTA: flags[i] is only ever written by this CTA
    closure_prepare<W>(n, list, i, sh);
    const uint32_t total = 1u << (sh.nfree > kClosureMaxFree ? kClosureMaxFree : sh.nfree);
    bool found = false;               // CTA-uniform: decided by a barrier vote, never read from shared memory
    for (uint32_t j0 = 0; j0 < total && !found; j0 += blockDim.x) {
      const uint32_t j = j0 + threadIdx.x;
      bool hit = false;
      if (j < total) {
        uint64_t t[W];
        closure_successor<W>(sh, j, t);
        const int64_t slot = hash_find<W>(t, tags, slot_state, cap_mask, injective);
        if (slot >= 0) {
          const unsigned long long k = slot_index[slot];
          hit = k != 0ull && reinterpret_cast<const volatile uint8_t*>(flags)[k - 1ull] != 0;
        }
      }
      found = __syncthreads_or(hit ? 1 : 0) != 0;
    }
    if (threadIdx.x == 0 && found) {
      flags[i] = 1;
      *changed = 1;
    }
    __syncthreads();                  // sh is rewritten by the next entry's closure_prepare
  }
}

}  // namespace pbn
