// Shared device-side definitions: kernel parameter block, table views, small helpers.
#pragma once
#ifndef __CUDACC_RTC__
#include <stdint.h>
#include <cuda_runtime.h>
#endif

#include "../../include/pbn_b200.h"
#include "philox.cuh"

namespace pbn {

// One predictor function, 16 bytes: 64-bit truth table (replicated over unused inputs, so a
// fixed-arity gather is branch-free) + 8 input gene indices.
struct __align__(16) FuncDesc {
  uint32_t lut_lo, lut_hi;
  uint32_t in03;  // inputs 0..3, one byte each
  uint32_t in47;  // inputs 4..7
};

// A wide predictor (arity 7..16): 16 input gene indices + where its truth table starts in wide_lut.
// Its FuncDesc carries in47 = kWideMarker (0xFF is never a gene index) and lut_lo = index into this table.
struct __align__(16) WideDesc {
  uint8_t in[16];
  uint32_t lut_off;   // in 64-bit words
  uint32_t arity;
  uint32_t pad[2];
};
constexpr uint32_t kWideMarker = 0xFFFFFFFFu;

// Everything a kernel needs besides the per-call arrays.  Passed by value (__grid_constant__).
struct NetParams {
  const int32_t* func_offset;   // [N+1]
  const FuncDesc* funcs;        // [F]
  const uint32_t* func_cum;     // [F]
  const uint32_t* survival;     // [N+1]
  const uint32_t* surv_sliced;  // [8N+1] survival table over the slots of one (column, warp) sub-stream
  const int32_t* attr_offset;   // [A+1]
  const uint64_t* attr_care;    // [S*W]
  const uint64_t* attr_val;     // [S*W]
  const uint32_t* pair_cum;     // [A*A] or nullptr
  int32_t n_genes, n_funcs, bins, horizon, pert_mode;
  int32_t n_attr, n_attr_states, pair_last;
  float r_success, r_step, r_action;
  uint32_t k0, k1;
  uint32_t sel_block_mask;      // bit b set: SELECT block b (genes 4b..4b+3) has a gene with >1 predictor
  uint32_t max_arity;
  uint32_t pert_rng;             // 1: draw perturbations from the stream (perturb_p > 0)
  uint32_t attr_simple;          // 1: every attractor is a single fully specified state (no wildcards)
  uint32_t rk[20];               // Philox round keys (k0 + r*W0, k1 + r*W1), r = 0..9: constant-bank operands
  float pert_inv_log2;           // 1 / log2(1 - perturb_p) (negative): first guess of the geometric skip
  const WideDesc* wide;          // [n_wide] or nullptr
  const uint64_t* wide_lut;      // multi-word truth tables of the wide predictors
  // Hash set over the fully specified attractor states (built by pbn_update_attractors for tables with large
  // attractors): open addressing, linear probing, key = the state, payload = its attractor.  nullptr: not built.
  const unsigned long long* ahash_tags;   // [mask + 1] fingerprint of the slot's state, 0 = empty
  const uint64_t* ahash_state;            // [(mask + 1) * W]
  const int32_t* ahash_attr;              // [mask + 1]
  const int32_t* awild_offset;            // [A + 1] CSR over the entries with wildcards ('*'), by attractor
  const int32_t* awild_entry;             // entry indices into attr_care / attr_val
  uint32_t ahash_mask;
  uint32_t awild_any;                     // some attractor has entries with wildcards (else the hash set alone decides)
  float r_wrong;                          // reward term for ending a step in a non-target attractor (0: not evaluated)
};

// Value of a wide predictor in state s (gather up to 16 state bits, look the bit up in global memory / L1).
template <int W>
__device__ __forceinline__ uint32_t eval_wide(const NetParams& n, uint32_t v, const uint64_t (&s)[W]) {
  const WideDesc wd = n.wide[v];
  uint32_t idx = 0;
  for (uint32_t j = 0; j < wd.arity; ++j) {
    const uint32_t g = wd.in[j];
    idx |= (uint32_t)((s[W == 1 ? 0 : (g >> 6)] >> (g & 63u)) & 1ull) << j;
  }
  return (uint32_t)(n.wide_lut[wd.lut_off + (idx >> 6)] >> (idx & 63u)) & 1u;
}

struct StepParams {
  pbn_step_args a;
  NetParams n;
  unsigned int* ticket;  // handle-owned; used to bump *a.step_ctr_dev once per launch
};

// pbn_rollout: n_steps uncontrolled updates with the state kept on chip in between.
struct RolloutParams {
  NetParams n;
  uint64_t* state;              // [E*W] in/out
  unsigned long long* stats;    // [PBN_N_STATS] or nullptr
  uint64_t step_ctr;            // Philox step counter of the first update
  int64_t env_offset, n_envs;
  int32_t n_steps;
};

// pbn_rollout_record: the rollout, and the states after every update s with s % stride == 0 counted into the caller's
// u64 accumulators (include/pbn_b200.h).
struct RecordParams {
  RolloutParams r;
  unsigned long long* gene_on;  // [N] or nullptr
  unsigned long long* hist;     // [2^n_proj] or nullptr
  int32_t stride, n_proj;
  int32_t proj[12];             // bin bit j = gene proj[j]
};

// Effective Philox step counter of this launch (host part + optional device-resident part).
__device__ __forceinline__ uint64_t effective_step(const pbn_step_args& a) {
  uint64_t step = a.step_ctr;
  if (a.step_ctr_dev != nullptr) step += *reinterpret_cast<const volatile uint64_t*>(a.step_ctr_dev);
  return step;
}

// Called by every thread at the very end of a step kernel: the last CTA to finish increments the
// device-resident step counter (every CTA read it before any CTA could get here last).
__device__ __forceinline__ void bump_device_step(const pbn_step_args& a, unsigned int* ticket) {
  if (a.step_ctr_dev == nullptr || (a.flags & (PBN_STEP_PDL | PBN_STEP_NO_COUNT))) return;
  // No fence is needed: the counter is only consumed by later launches (ordered by the stream),
  // and every thread of this CTA has used its copy of the counter before the barrier below.
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(ticket, 1u);
    if (t == gridDim.x - 1) {
      *ticket = 0;
      *a.step_ctr_dev += 1;
    }
  }
}

// Dynamic shared-memory layout of the sliced kernel (computed by the host per launch).
struct SlicedSmemLayout {
  uint32_t surv_off, rew_off, aoffs_off, acare_off, aval_off, scratch_off, total;
  uint32_t stage_state_off, stage_act_off, mbar_off;  // TMA staging of a tile's state / action bytes
  uint32_t attractors_in_smem;
  // pbn_step_sliced_gen with the hash set: per attractor its FIRST entry ([care | value] at acare_off, as in the
  // single-state layout) and its number of entries (at aoffs_off) -- single-state targets are then tested in shared
  // memory and only the envs whose target is a larger attractor probe the hash set
  uint32_t singles_in_smem;
};

// Dynamic shared-memory layout of the plane-resident kernel's attractor tables (byte offsets; the fixed part of
// the layout is compile-time, step_planes.cuh).
struct PlanesLayout {
  uint32_t aval_off, acare_off, aoffs_off, eattr_off, total;
  uint32_t attr_in_smem;
};

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// number of entries k in the non-increasing table tab[1..n] with u < tab[k]   (geometric skip)
__device__ __forceinline__ int count_below_survival(const uint32_t* tab, int n, uint32_t u) {
  int lo = 0, hi = n;  // invariant: u < tab[lo] (tab[0] = 2^32 conceptually), !(u < tab[hi+1])
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (u < tab[mid]) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// number of entries k in [0, n) of the non-decreasing table with tab[k] <= u
__device__ __forceinline__ int count_le(const uint32_t* tab, int n, uint32_t u) {
  int lo = 0, hi = n;  // answer in [lo, hi]
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (tab[mid] <= u) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// (source, target) pair of env.reset() from word 0 of the env's RESET block.
__device__ __forceinline__ void reset_pair(const NetParams& n, const Philox4& r, int& src, int& tgt) {
  const int A = n.n_attr;
  if (n.pair_cum != nullptr) {
    int pair = count_le(n.pair_cum, A * A - 1, r.x);
    pair = min(pair, n.pair_last);
    src = pair / A;
    tgt = pair - src * A;
  } else if (A > 1) {
    // q = floor(x A (A-1) / 2^32), src = floor(q / (A-1)) = floor(x A / 2^32): no integer division needed
    const uint32_t q = __umulhi(r.x, (uint32_t)(A * (A - 1)));
    src = (int)__umulhi(r.x, (uint32_t)A);
    const int tt = (int)(q - (uint32_t)src * (uint32_t)(A - 1));
    tgt = tt + (tt >= src ? 1 : 0);
  } else {
    src = 0;
    tgt = 0;
  }
}

// (source, target) draw + source state for env.reset(); r = Philox block (RESET, 0) of the env.
template <int W>
__device__ __forceinline__ void reset_draw(const NetParams& n, const Philox4& r, uint64_t (&s)[W], int& src,
                                           int& tgt) {
  const int A = n.n_attr;
  if (n.pair_cum != nullptr) {
    int pair = count_le(n.pair_cum, A * A - 1, r.x);
    pair = min(pair, n.pair_last);
    src = pair / A;
    tgt = pair - src * A;
  } else if (A > 1) {
    // q = floor(x A (A-1) / 2^32), src = floor(q / (A-1)) = floor(x A / 2^32): no integer division needed
    const uint32_t q = __umulhi(r.x, (uint32_t)(A * (A - 1)));
    src = (int)__umulhi(r.x, (uint32_t)A);
    const int tt = (int)(q - (uint32_t)src * (uint32_t)(A - 1));
    tgt = tt + (tt >= src ? 1 : 0);
  } else {
    src = 0;
    tgt = 0;
  }
  const int o0 = n.attr_offset[src];
  const int ns = n.attr_offset[src + 1] - o0;
  const int j = o0 + (int)__umulhi(r.y, (uint32_t)ns);
#pragma unroll
  for (int w = 0; w < W; ++w) s[w] = n.attr_val[(size_t)j * W + w];
}

// splitmix64 finaliser; shared by the attractor hash set and the visit-count table (discover.cuh)
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) {
  x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27; x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return x;
}

// Fingerprint of a state in the attractor hash set: never 0 (an empty slot).  The host builds the table with the
// same function (pbn_update_attractors).
__host__ __device__ __forceinline__ uint64_t attr_tag(const uint64_t* s, int W) {
  uint64_t h = mix64(s[0] + 0x9E3779B97F4A7C15ull);
  if (W == 2) h = mix64(h ^ (s[1] + 0xD1B54A32D192ED03ull));
  return h == 0ull ? 1ull : h;
}

// Home slot of a fingerprint: its upper half (the fingerprint is a splitmix64 output -- mixing it a second time bought
// nothing and cost the step kernels as much as the fingerprint itself).
__host__ __device__ __forceinline__ uint32_t attr_slot(uint64_t tag, uint32_t mask) { return (uint32_t)(tag >> 32) & mask; }

// env.in_target(state) through the hash set: is `s` a state of attractor `a`?  O(1) expected: one probe sequence over
// the fully specified states (tag match confirmed on the state words and the attractor id) + the attractor's few
// wildcard entries.  model_tester.py:602-616; bdq_model/__init__.py:182-184 (attractor sets that grow).
template <int W>
__device__ __forceinline__ bool in_attractor_hashed(const NetParams& n, int a, const uint64_t (&s)[W]) {
  const uint64_t tag = attr_tag(s, W);
  uint32_t slot = attr_slot(tag, n.ahash_mask);
  for (uint32_t probe = 0; probe <= n.ahash_mask; ++probe, slot = (slot + 1u) & n.ahash_mask) {
    const unsigned long long cur = n.ahash_tags[slot];
    if (cur == 0ull) break;
    if (cur == tag && n.ahash_attr[slot] == a) {
      bool same = true;
#pragma unroll
      for (int w = 0; w < W; ++w) same = same && n.ahash_state[(size_t)slot * W + w] == s[w];
      if (same) return true;
    }
  }
  for (int k = n.awild_offset[a]; k < n.awild_offset[a + 1]; ++k) {
    const int e = n.awild_entry[k];
    bool m = true;
#pragma unroll
    for (int w = 0; w < W; ++w) m = m && ((s[w] & n.attr_care[(size_t)e * W + w]) == n.attr_val[(size_t)e * W + w]);
    if (m) return true;
  }
  return false;
}

// env.state_attractor_id through the hash set: the first (lowest-numbered) attractor containing `s`, or -1.
template <int W>
__device__ __forceinline__ int attractor_of_hashed(const NetParams& n, const uint64_t (&s)[W]) {
  int best = n.n_attr;
  const uint64_t tag = attr_tag(s, W);
  uint32_t slot = attr_slot(tag, n.ahash_mask);
  for (uint32_t probe = 0; probe <= n.ahash_mask; ++probe, slot = (slot + 1u) & n.ahash_mask) {
    const unsigned long long cur = n.ahash_tags[slot];
    if (cur == 0ull) break;
    if (cur == tag && n.ahash_attr[slot] < best) {
      bool same = true;
#pragma unroll
      for (int w = 0; w < W; ++w) same = same && n.ahash_state[(size_t)slot * W + w] == s[w];
      if (same) best = n.ahash_attr[slot];
    }
  }
  for (int a = 0; a < best; ++a)
    for (int k = n.awild_offset[a]; k < n.awild_offset[a + 1]; ++k) {
      const int e = n.awild_entry[k];
      bool m = true;
#pragma unroll
      for (int w = 0; w < W; ++w) m = m && ((s[w] & n.attr_care[(size_t)e * W + w]) == n.attr_val[(size_t)e * W + w]);
      if (m) { best = a; break; }
    }
  return best < n.n_attr ? best : -1;
}

// "wrong attractor" test of the reward (r_wrong != 0): s lies in some attractor other than `target`
template <int W>
__device__ __forceinline__ bool in_other_attractor(const NetParams& n, int target, const uint64_t (&s)[W]);

template <int W>
__device__ __forceinline__ bool in_attractor(const int32_t* offs, const uint64_t* care, const uint64_t* val,
                                             int a, const uint64_t (&s)[W]) {
  bool hit = false;
  const int e1 = offs[a + 1];
  for (int e = offs[a]; e < e1; ++e) {
    bool m = true;
#pragma unroll
    for (int w = 0; w < W; ++w) m = m && ((s[w] & care[(size_t)e * W + w]) == val[(size_t)e * W + w]);
    hit = hit || m;
  }
  return hit;
}

template <int W>
__device__ __forceinline__ bool in_other_attractor(const NetParams& n, int target, const uint64_t (&s)[W]) {
  if (n.ahash_tags != nullptr) {
    const int a = attractor_of_hashed<W>(n, s);   // the lowest-numbered attractor holding s; a state of the target is a hit, not a miss
    return a >= 0 && a != target;
  }
  for (int a = 0; a < n.n_attr; ++a)
    if (a != target && in_attractor<W>(n.attr_offset, n.attr_care, n.attr_val, a, s)) return true;
  return false;
}

}  // namespace pbn
