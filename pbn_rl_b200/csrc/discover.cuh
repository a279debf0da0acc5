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

// ---- exhaustive attractor search: backward reachability over every state (N <= PBN_DP_MAX_GENES) ----
// marks holds one bit per state (bit s & 31 of word s >> 5).  The caller marks the states of the attractors known so
// far (reach_mark_kernel); a sweep then marks every unmarked state one of whose successors is marked, and the caller
// repeats sweeps until one marks nothing.  The result is the set of states that reach a known attractor -- the least
// fixed point, whatever order the bits land in: a bit set early in a sweep may be seen later in the same sweep, which
// only saves sweeps.  At p = 0 every state reaches a sink SCC and sink SCCs are closed, so a fixed point with every bit
// set proves that the known attractors are all of them.  Successors are those of the perturbation-free STG, the
// relation of successor_descriptor: a gene is free when some predictor yields 1 and some yields 0.

// The valid state bits of a marks word: all 32, or the 2^N of the single partial word when N < 5.
__device__ __forceinline__ uint32_t reach_valid_bits(int n_genes) {
  return n_genes >= 5 ? 0xFFFFFFFFu : (1u << (1u << n_genes)) - 1u;
}

// One warp per marks word (32 states), words [w0, w0 + count); a word whose valid bits are all set is skipped.  For
// each unmarked state s of the word, lane g < N evaluates gene g's predictors and two ballots give the fixed genes and
// the free ones.  The free genes split into L (genes 0..4, inside one marks word) and H (genes 5 and up, which pick the
// word): a successor t lies in word ((fixed | c) >> 5) for c a subset of H, at a bit of the mask M (lane b of a third
// ballot: (b ^ fixed) & 31 & ~L == 0).  The lanes walk those 2^|H| words 32 at a time -- lane l takes the subset of
// H's five lowest genes given by the bits of l, the remaining genes of H advance in the loop -- and stop at the first
// word with a marked bit under M.  *newly gains the number of bits the sweep set.
__global__ void __launch_bounds__(256) reach_sweep_kernel(const __grid_constant__ NetParams n, uint32_t* __restrict__ marks,
                                                          uint32_t w0, uint32_t count,
                                                          unsigned long long* __restrict__ newly) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t valid = reach_valid_bits(n.n_genes);
  uint32_t set = 0;   // bits this warp set (counted by lane 0)
  for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < count; i += (gridDim.x * blockDim.x) >> 5) {
    const uint32_t w = w0 + i;
    uint32_t todo = __shfl_sync(0xFFFFFFFFu, lane == 0 ? ~__ldcg(marks + w) & valid : 0u, 0);
    while (todo) {
      const uint32_t b = __ffs(todo) - 1;
      todo &= todo - 1u;
      const uint32_t s = (w << 5) | b;
      bool can1 = false, can0 = false;
      if ((int)lane < n.n_genes) {
        const uint64_t st[1] = {s};
        for (int f = n.func_offset[lane]; f < n.func_offset[lane + 1]; ++f) {
          if (eval_func<1>(n, f, st)) can1 = true; else can0 = true;
        }
      }
      const uint32_t one = __ballot_sync(0xFFFFFFFFu, can1), zero = __ballot_sync(0xFFFFFFFFu, can0);
      const uint32_t fr = one & zero, fixed = one & ~zero;
      const uint32_t m = __ballot_sync(0xFFFFFFFFu, ((lane ^ fixed) & 31u & ~fr) == 0u);
      const uint32_t base = fixed >> 5, hw = fr >> 5;   // word index: base | (a subset of hw); base & hw = 0
      uint32_t hhi = hw, clo = 0;
      int k = 0;
      for (; k < 5 && hhi; ++k) {
        const uint32_t g = hhi & (0u - hhi);
        hhi ^= g;
        if ((lane >> k) & 1u) clo |= g;
      }
      const bool active = (lane >> k) == 0u;
      bool hit = false;
      uint32_t chi = 0;
      do {
        hit = __any_sync(0xFFFFFFFFu, active && (__ldcg(marks + (base | clo | chi)) & m) != 0u);
        chi = (chi - hhi) & hhi;   // the next subset of hhi in increasing order; 0 again after the last
      } while (!hit && chi != 0u);
      if (hit && lane == 0) {
        const uint32_t bit = 1u << b;
        if (!(atomicOr(marks + w, bit) & bit)) ++set;
      }
    }
  }
  if (lane == 0 && set != 0u) atomicAdd(newly, (unsigned long long)set);
}

// Set the bits of states[0, n_states); states >= n_valid (= 2^N) are ignored.  *newly gains the number of bits set.
__global__ void __launch_bounds__(256) reach_mark_kernel(uint32_t* __restrict__ marks, const uint64_t* __restrict__ states,
                                                         int64_t n_states, uint64_t n_valid,
                                                         unsigned long long* __restrict__ newly) {
  uint32_t set = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_states; i += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t s = states[i];
    if (s >= n_valid) continue;
    const uint32_t bit = 1u << (s & 31u);
    if (!(atomicOr(marks + (s >> 5), bit) & bit)) ++set;
  }
  set = __reduce_add_sync(0xFFFFFFFFu, set);
  if ((threadIdx.x & 31u) == 0 && set != 0u) atomicAdd(newly, (unsigned long long)set);
}

}  // namespace pbn
