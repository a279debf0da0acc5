// pbn_record_states: steady-state statistics of row-format states (any kernel) -- per-gene ON counts and a histogram of
// the states projected onto up to 12 genes, added into caller-owned u64 accumulators (include/pbn_b200.h).  The
// policy-in-the-loop form of compute_ssd_hist (train_pbn_28.py:257) records after every pbn_step with this; the
// uncontrolled form records inside the rollout (step_sliced.cuh, pbn_rollout_sliced<true>).
#pragma once
#include "pbn_common.cuh"

namespace pbn {

constexpr int kRecordThreads = 256;

struct RecordStatesParams {
  const uint64_t* state;           // [E*W]
  unsigned long long* gene_on;     // [N] or nullptr
  unsigned long long* hist;        // [2^n_proj] or nullptr
  int64_t n_envs;
  int32_t n_genes, W, n_proj;
  int32_t proj[12];                // bin bit j = gene proj[j]
};

// Grid-stride over warps of 32 envs (one env per lane).  Gene g: one ballot over the warp, counted by lane g mod 32 in
// a register.  Histogram: u32 bins in shared memory; the lanes that share a bin add once.  A block covers at most
// ceil(E / grid) + 256 envs; with grid = min(ceil(E / 256), 4 * #SMs) that stays below 2^32 for every batch whose
// state array fits in device memory (2^32 * 4 * 148 envs would take 20 TB), so the u32 bins cannot overflow.
__global__ void __launch_bounds__(kRecordThreads) record_states_kernel(const __grid_constant__ RecordStatesParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* s_gene = reinterpret_cast<unsigned long long*>(smem_raw);   // [128]
  uint32_t* bins = reinterpret_cast<uint32_t*>(smem_raw + 128 * sizeof(unsigned long long));
  const int nbins = p.hist != nullptr ? 1 << p.n_proj : 0;
  const uint32_t lane = threadIdx.x & 31u;
  for (int i = threadIdx.x; i < 128; i += kRecordThreads) s_gene[i] = 0ull;
  for (int b = threadIdx.x; b < nbins; b += kRecordThreads) bins[b] = 0u;
  __syncthreads();
  unsigned long long cnt[4] = {0ull, 0ull, 0ull, 0ull};   // genes lane, lane + 32, lane + 64, lane + 96
  const int64_t warps = (int64_t)gridDim.x * (kRecordThreads / 32);
  for (int64_t base = ((int64_t)blockIdx.x * (kRecordThreads / 32) + (threadIdx.x >> 5)) * 32; base < p.n_envs; base += warps * 32) {
    const int64_t e = base + lane;
    const bool ok = e < p.n_envs;
    uint64_t s0 = 0ull, s1 = 0ull;
    if (ok) {
      s0 = p.state[e * p.W];
      if (p.W > 1) s1 = p.state[e * p.W + 1];
    }
    if (p.gene_on != nullptr) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint64_t sw = k < 2 ? s0 : s1;
        for (int gl = 0; gl < 32 && 32 * k + gl < p.n_genes; ++gl) {
          const uint32_t b = __ballot_sync(0xFFFFFFFFu, (sw >> (32 * (k & 1) + gl)) & 1ull);   // padding lanes hold 0
          if ((uint32_t)gl == lane) cnt[k] += (unsigned long long)__popc(b);
        }
      }
    }
    if (p.hist != nullptr) {
      uint32_t idx = 0u;
      for (int j = 0; j < p.n_proj; ++j) {
        const int g = p.proj[j];
        idx |= (uint32_t)(((g < 64 ? s0 : s1) >> (g & 63)) & 1ull) << j;
      }
      const uint32_t peers = __match_any_sync(0xFFFFFFFFu, ok ? idx : 0xFFFFFFFFu);
      if (ok && __ffs(peers) - 1 == (int)lane) atomicAdd(&bins[idx], (uint32_t)__popc(peers));
    }
  }
  if (p.gene_on != nullptr) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (cnt[k] != 0ull) atomicAdd(&s_gene[32 * k + lane], cnt[k]);
  }
  __syncthreads();
  if (p.gene_on != nullptr)
    for (int g = threadIdx.x; g < p.n_genes; g += kRecordThreads)
      if (s_gene[g] != 0ull) atomicAdd(&p.gene_on[g], s_gene[g]);
  for (int b = threadIdx.x; b < nbins; b += kRecordThreads)
    if (bins[b] != 0u) atomicAdd(&p.hist[b], (unsigned long long)bins[b]);
}

}  // namespace pbn
