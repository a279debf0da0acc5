// Scalar ("thread-per-env") step kernel: the general path.
//
// One thread owns one env instance for the whole step: packed state in registers, the
// network's truth tables (FuncDesc) + selection thresholds + survival table + (if small)
// the attractor table staged once per CTA into shared memory.  Handles any network the ABI
// admits (N <= 128, arity <= 6, any number of predictors per gene with arbitrary
// selection probabilities).  HBM access is coalesced: consecutive lanes own consecutive envs.
//
// Algorithmic HBM bytes per env-step (N <= 64, bins = 3): state 8 r + 8 w, actions 3 r,
// target id 4 r, t 2 r + 2 w, reward 4 w, terminated 1 w, truncated 1 w = 33 B.
#pragma once
#include "pbn_common.cuh"

namespace pbn {

struct ScalarSmemLayout {
  uint32_t funcs_off, offs_off, cum_off, surv_off, aoffs_off, acare_off, aval_off, total;
  bool attractors_in_smem;
};

inline ScalarSmemLayout scalar_smem_layout(const NetParams& n, int W) {
  ScalarSmemLayout L{};
  uint32_t o = 0;
  L.funcs_off = o; o += (uint32_t)n.n_funcs * 16u;
  L.offs_off = o;  o += (uint32_t)(n.n_genes + 1) * 4u;
  L.cum_off = o;   o += (uint32_t)n.n_funcs * 4u;
  L.surv_off = o;  o += (uint32_t)(n.n_genes + 1) * 4u;
  o = (o + 15u) & ~15u;
  const uint32_t abytes = (uint32_t)(n.n_attr + 1) * 4u + (uint32_t)n.n_attr_states * W * 16u + 32u;
  L.attractors_in_smem = n.n_attr > 0 && abytes <= 32u * 1024u;
  if (L.attractors_in_smem) {
    L.acare_off = o; o += (uint32_t)n.n_attr_states * W * 8u;
    L.aval_off = o;  o += (uint32_t)n.n_attr_states * W * 8u;
    L.aoffs_off = o; o += (uint32_t)(n.n_attr + 1) * 4u;
    o = (o + 15u) & ~15u;
  }
  L.total = o;
  return L;
}

template <int W>
__device__ __forceinline__ uint32_t state_bit(const uint64_t (&s)[W], uint32_t g) {
  if constexpr (W == 1) {
    return (uint32_t)(s[0] >> g) & 1u;
  } else {
    const uint64_t w = (g & 64u) ? s[1] : s[0];
    return (uint32_t)(w >> (g & 63u)) & 1u;
  }
}

// MAXA = 4: truth tables are 16-bit (replicated), 4 gathers per gene; MAXA = 6: 64-bit, 6 gathers;
// MAXA = 16: as 6, plus wide predictors (multi-word tables in global memory).
template <int W, int MAXA>
__global__ void __launch_bounds__(256) step_scalar_kernel(const __grid_constant__ StepParams p,
                                                         const ScalarSmemLayout L) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const NetParams& n = p.n;
  const pbn_step_args& a = p.a;
  FuncDesc* s_funcs = reinterpret_cast<FuncDesc*>(smem_raw + L.funcs_off);
  int32_t* s_offs = reinterpret_cast<int32_t*>(smem_raw + L.offs_off);
  uint32_t* s_cum = reinterpret_cast<uint32_t*>(smem_raw + L.cum_off);
  uint32_t* s_surv = reinterpret_cast<uint32_t*>(smem_raw + L.surv_off);
  uint64_t* s_acare = reinterpret_cast<uint64_t*>(smem_raw + L.acare_off);
  uint64_t* s_aval = reinterpret_cast<uint64_t*>(smem_raw + L.aval_off);
  int32_t* s_aoffs = reinterpret_cast<int32_t*>(smem_raw + L.aoffs_off);

  for (int i = threadIdx.x; i < n.n_funcs; i += blockDim.x) {
    s_funcs[i] = n.funcs[i];
    s_cum[i] = n.func_cum[i];
  }
  for (int i = threadIdx.x; i <= n.n_genes; i += blockDim.x) {
    s_offs[i] = n.func_offset[i];
    s_surv[i] = n.survival[i];
  }
  if (L.attractors_in_smem) {
    for (int i = threadIdx.x; i < n.n_attr_states * W; i += blockDim.x) {
      s_acare[i] = n.attr_care[i];
      s_aval[i] = n.attr_val[i];
    }
    for (int i = threadIdx.x; i <= n.n_attr; i += blockDim.x) s_aoffs[i] = n.attr_offset[i];
  }
  __syncthreads();
  const int32_t* aoffs = L.attractors_in_smem ? s_aoffs : n.attr_offset;
  const uint64_t* acare = L.attractors_in_smem ? s_acare : n.attr_care;
  const uint64_t* aval = L.attractors_in_smem ? s_aval : n.attr_val;

  const int N = n.n_genes;
  const bool injected = a.sel != nullptr;
  const uint64_t step_ctr = effective_step(a);
  unsigned long long st_eps = 0, st_term = 0, st_trunc = 0, st_len = 0, st_flips = 0, st_pert = 0, st_steps = 0;

  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < a.n_envs;
       e += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t gid = (uint64_t)(a.env_offset + e);
    uint64_t s[W];
#pragma unroll
    for (int w = 0; w < W; ++w) s[w] = a.state[e * W + w];

    // 1. interventions
    uint64_t flip[W];
#pragma unroll
    for (int w = 0; w < W; ++w) flip[w] = 0;
    if (a.actions != nullptr) {
      for (int j = 0; j < n.bins; ++j) {
        const uint32_t act = a.actions[e * n.bins + j];
        if (act >= 1u && act <= (uint32_t)N) {
          const uint32_t g = act - 1u;
          if constexpr (W == 1) flip[0] |= 1ull << g;
          else flip[g >> 6] |= 1ull << (g & 63u);
        }
      }
    }
    int nflips = 0;
#pragma unroll
    for (int w = 0; w < W; ++w) {
      s[w] ^= flip[w];
      nflips += __popcll(flip[w]);
    }

    // 2+3. predictor selection and synchronous update
    uint64_t f[W];
#pragma unroll
    for (int w = 0; w < W; ++w) f[w] = 0;
    Philox4 rb{0, 0, 0, 0};
    for (int i = 0; i < N; ++i) {
      const int fo = s_offs[i];
      const int K = s_offs[i + 1] - fo;
      int k = 0;
      if (injected) {
        k = a.sel[e * N + i];
        k = k < K ? k : K - 1;
      } else {
        if ((i & 3) == 0 && ((n.sel_block_mask >> (i >> 2)) & 1u))
          rb = philox_stream(gid, step_ctr, PBN_RNG_SELECT, (uint32_t)(i >> 2), n.k0, n.k1);
        if (K > 1) {
          const uint32_t u = (i & 3) == 0 ? rb.x : (i & 3) == 1 ? rb.y : (i & 3) == 2 ? rb.z : rb.w;
          for (int c = 0; c < K - 1; ++c) k += (s_cum[fo + c] <= u) ? 1 : 0;
        }
      }
      const FuncDesc fd = s_funcs[fo + k];
      uint32_t idx = 0;
      uint32_t bit;
      if (MAXA > 6 && fd.in47 == kWideMarker) {
        bit = eval_wide<W>(n, fd.lut_lo, s);
        if constexpr (W == 1) f[0] |= (uint64_t)bit << i;
        else f[i >> 6] |= (uint64_t)bit << (i & 63);
        continue;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) idx |= state_bit<W>(s, (fd.in03 >> (8 * j)) & 0xFFu) << j;
      if constexpr (MAXA == 4) {
        bit = (fd.lut_lo >> idx) & 1u;
      } else {
#pragma unroll
        for (int j = 0; j < 2; ++j) idx |= state_bit<W>(s, (fd.in47 >> (8 * j)) & 0xFFu) << (4 + j);
        const uint64_t lut = ((uint64_t)fd.lut_hi << 32) | fd.lut_lo;
        bit = (uint32_t)(lut >> idx) & 1u;
      }
      if constexpr (W == 1) f[0] |= (uint64_t)bit << i;
      else f[i >> 6] |= (uint64_t)bit << (i & 63);
    }

    // 4. perturbation
    uint64_t pert[W];
#pragma unroll
    for (int w = 0; w < W; ++w) pert[w] = 0;
    if (n.pert_mode != PBN_PERT_NONE) {
      if (injected) {
        if (a.pert_mask != nullptr) {
#pragma unroll
          for (int w = 0; w < W; ++w) pert[w] = a.pert_mask[e * W + w];
        }
      } else if (n.pert_rng) {
        int pos = -1;
        uint32_t draw = 0;
        Philox4 pb{0, 0, 0, 0};
        while (true) {
          if ((draw & 3u) == 0u) pb = philox_stream(gid, step_ctr, PBN_RNG_PERTURB, draw >> 2, n.k0, n.k1);
          const uint32_t u = (draw & 3u) == 0 ? pb.x : (draw & 3u) == 1 ? pb.y : (draw & 3u) == 2 ? pb.z : pb.w;
          ++draw;
          pos += count_below_survival(s_surv, N, u) + 1;
          if (pos >= N) break;
          if constexpr (W == 1) pert[0] |= 1ull << pos;
          else pert[pos >> 6] |= 1ull << (pos & 63);
        }
      }
    }
    uint64_t nx[W];
    bool any_pert = false;
#pragma unroll
    for (int w = 0; w < W; ++w) any_pert = any_pert || (pert[w] != 0);
#pragma unroll
    for (int w = 0; w < W; ++w) {
      if (n.pert_mode == PBN_PERT_A) nx[w] = any_pert ? (s[w] ^ pert[w]) : f[w];
      else if (n.pert_mode == PBN_PERT_B) nx[w] = f[w] ^ pert[w];
      else if (n.pert_mode == PBN_PERT_C) nx[w] = (f[w] & ~pert[w]) | (~s[w] & pert[w]);
      else nx[w] = f[w];
    }
    if (n.pert_mode == PBN_PERT_C) {  // ~s1 may set bits above N
      if constexpr (W == 1) nx[0] &= (N == 64) ? ~0ull : ((1ull << N) - 1ull);
      else nx[1] &= (N == 128) ? ~0ull : ((1ull << (N - 64)) - 1ull);
    }

    // 5-7. target test, counters, reward
    bool hit = false;
    int tgt = -1;
    if (a.target_id != nullptr) {
      tgt = a.target_id[e];
      if (tgt >= 0 && tgt < n.n_attr) hit = n.ahash_tags != nullptr ? in_attractor_hashed<W>(n, tgt, nx) : in_attractor<W>(aoffs, acare, aval, tgt, nx);
    }
    uint32_t tt = a.t != nullptr ? a.t[e] : 0u;
    tt = tt < 65535u ? tt + 1u : 65535u;
    const bool trunc = !hit && n.horizon > 0 && tt >= (uint32_t)n.horizon;
    const float base = __fadd_rn(n.r_step, __fmul_rn(n.r_action, (float)nflips));
    float bonus = hit ? n.r_success : 0.0f;
    if (!hit && n.r_wrong != 0.0f && n.n_attr > 0 && in_other_attractor<W>(n, tgt, nx)) bonus = n.r_wrong;
    const float rew = __fadd_rn(base, bonus);
    if (a.reward != nullptr) a.reward[e] = rew;
    if (a.terminated != nullptr) a.terminated[e] = hit ? 1 : 0;
    if (a.truncated != nullptr) a.truncated[e] = trunc ? 1 : 0;
    if (a.final_state != nullptr) {
#pragma unroll
      for (int w = 0; w < W; ++w) a.final_state[e * W + w] = nx[w];
    }
    const bool done = hit || trunc;
    st_steps += 1;
    st_flips += nflips;
#pragma unroll
    for (int w = 0; w < W; ++w) st_pert += __popcll(pert[w]);
    if (done) {
      st_eps += 1;
      st_term += hit ? 1 : 0;
      st_trunc += trunc ? 1 : 0;
      st_len += tt;
    }

    // 8. auto-reset
    if (done && (a.flags & PBN_STEP_AUTORESET)) {
      const Philox4 r = philox_stream(gid, step_ctr, PBN_RNG_RESET, 0, n.k0, n.k1);
      int src;
      reset_draw<W>(n, r, nx, src, tgt);
      a.target_id[e] = tgt;
      if (a.source_id != nullptr) a.source_id[e] = src;
      tt = 0;
    }
#pragma unroll
    for (int w = 0; w < W; ++w) a.state[e * W + w] = nx[w];
    if (a.t != nullptr) a.t[e] = (uint16_t)tt;
  }

  if (a.stats != nullptr) {
    unsigned long long v[7] = {st_steps, st_eps, st_term, st_trunc, st_len, st_flips, st_pert};
#pragma unroll
    for (int q = 0; q < 7; ++q) {
      unsigned long long x = v[q];
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, d);
      if (lane_id() == 0 && x != 0) atomicAdd(&a.stats[q], x);
    }
  }
  bump_device_step(a, p.ticket);
}

// ------------------------------------------------------------------------------------------
// small companions
// ------------------------------------------------------------------------------------------

template <int W>
__global__ void __launch_bounds__(256) reset_kernel(const __grid_constant__ NetParams n, uint64_t* state,
                                                   int32_t* target_id, int32_t* source_id, uint16_t* t,
                                                   const uint8_t* done_mask, uint64_t step_ctr,
                                                   int64_t env_offset, int64_t n_envs) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_envs;
       e += (int64_t)gridDim.x * blockDim.x) {
    if (done_mask != nullptr && done_mask[e] == 0) continue;
    const Philox4 r = philox_stream((uint64_t)(env_offset + e), step_ctr, PBN_RNG_RESET, 0, n.k0, n.k1);
    uint64_t s[W];
    int src, tgt;
    reset_draw<W>(n, r, s, src, tgt);
#pragma unroll
    for (int w = 0; w < W; ++w) state[e * W + w] = s[w];
    if (target_id != nullptr) target_id[e] = tgt;
    if (source_id != nullptr) source_id[e] = src;
    if (t != nullptr) t[e] = 0;
  }
}

__global__ void advance_counter_kernel(uint64_t* ctr, uint64_t n) { *ctr += n; }

// pbn_step_host: stream one lane's results from the device arrays into page-locked host memory that
// is mapped into the device address space (zero-copy posted writes over PCIe, 16 B per thread).
// A few CTAs saturate the link (scripts/micro/zerocopy_rate.cu); the grid is kept small so that the
// step kernels of the other lanes find free SMs.
struct ExportArgs {
  const uint8_t* src[4];
  uint8_t* dst[4];
  unsigned long long bytes[4];
  // compact outputs (optional): state narrowed to 32 bits (N <= 32), done = terminated | truncated << 1
  const uint64_t* state64;
  uint32_t* state32;
  const uint8_t* term;
  const uint8_t* trunc;
  uint8_t* done;
  uint32_t* packed;   // state | terminated << 30 | truncated << 31 (N <= 30)
  long long n_envs;
};

// actions16[e] = a0 | a1 << 5 | a2 << 10  ->  the 3 action bytes of env e (four envs per thread)
__global__ void __launch_bounds__(256) unpack_actions16_kernel(const uint16_t* __restrict__ a16, uint8_t* __restrict__ out, long long n_envs) {
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
  const size_t n4 = (size_t)n_envs >> 2;
  const bool vec = ((reinterpret_cast<uintptr_t>(a16) & 7u) | (reinterpret_cast<uintptr_t>(out) & 3u)) == 0;
  if (vec) {
    for (size_t i = tid; i < n4; i += nth) {
      const uint2 v = reinterpret_cast<const uint2*>(a16)[i];
      uint32_t b[12];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const uint32_t x = ((e < 2 ? v.x : v.y) >> (16 * (e & 1))) & 0xFFFFu;
        b[3 * e] = x & 31u; b[3 * e + 1] = (x >> 5) & 31u; b[3 * e + 2] = (x >> 10) & 31u;
      }
#pragma unroll
      for (int q = 0; q < 3; ++q)
        reinterpret_cast<uint32_t*>(out)[3 * i + q] = b[4 * q] | (b[4 * q + 1] << 8) | (b[4 * q + 2] << 16) | (b[4 * q + 3] << 24);
    }
  }
  for (size_t e = (vec ? (n4 << 2) : 0) + tid; e < (size_t)n_envs; e += nth) {
    const uint32_t x = a16[e];
    out[3 * e] = (uint8_t)(x & 31u); out[3 * e + 1] = (uint8_t)((x >> 5) & 31u); out[3 * e + 2] = (uint8_t)((x >> 10) & 31u);
  }
}

__global__ void __launch_bounds__(256) export_kernel(ExportArgs x) {
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint8_t* __restrict__ src = x.src[k];
    uint8_t* __restrict__ dst = x.dst[k];
    const size_t nb = x.bytes[k];
    if (dst == nullptr || nb == 0) continue;
    if (((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 15u) != 0) {
      for (size_t i = tid; i < nb; i += nth) dst[i] = src[i];
      continue;
    }
    const size_t nv = nb >> 4;
    for (size_t i = tid; i < nv; i += nth) reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(src)[i];
    for (size_t i = (nv << 4) + tid; i < nb; i += nth) dst[i] = src[i];
  }
  // compact forms, four envs per thread and iteration: one 16 B / one 4 B posted write each
  const size_t n4 = (size_t)x.n_envs >> 2;
  if (x.state32 != nullptr) {
    const bool vec = ((reinterpret_cast<uintptr_t>(x.state64) | reinterpret_cast<uintptr_t>(x.state32)) & 15u) == 0;
    if (vec) {
      for (size_t i = tid; i < n4; i += nth) {
        const uint4 a = reinterpret_cast<const uint4*>(x.state64)[2 * i], b = reinterpret_cast<const uint4*>(x.state64)[2 * i + 1];
        reinterpret_cast<uint4*>(x.state32)[i] = make_uint4(a.x, a.z, b.x, b.z);
      }
    }
    for (size_t e = (vec ? (n4 << 2) : 0) + tid; e < (size_t)x.n_envs; e += nth) x.state32[e] = (uint32_t)x.state64[e];
  }
  if (x.packed != nullptr) {
    const bool vec = ((reinterpret_cast<uintptr_t>(x.state64) | reinterpret_cast<uintptr_t>(x.packed)) & 15u) == 0 &&
                     ((reinterpret_cast<uintptr_t>(x.term) | reinterpret_cast<uintptr_t>(x.trunc)) & 3u) == 0;
    if (vec) {
      for (size_t i = tid; i < n4; i += nth) {
        const uint4 a = reinterpret_cast<const uint4*>(x.state64)[2 * i], b = reinterpret_cast<const uint4*>(x.state64)[2 * i + 1];
        const uint32_t te = reinterpret_cast<const uint32_t*>(x.term)[i], tr = reinterpret_cast<const uint32_t*>(x.trunc)[i];
        reinterpret_cast<uint4*>(x.packed)[i] =
            make_uint4(a.x | ((te & 1u) << 30) | ((tr & 1u) << 31), a.z | (((te >> 8) & 1u) << 30) | (((tr >> 8) & 1u) << 31),
                       b.x | (((te >> 16) & 1u) << 30) | (((tr >> 16) & 1u) << 31), b.z | (((te >> 24) & 1u) << 30) | (((tr >> 24) & 1u) << 31));
      }
    }
    for (size_t e = (vec ? (n4 << 2) : 0) + tid; e < (size_t)x.n_envs; e += nth)
      x.packed[e] = (uint32_t)x.state64[e] | ((uint32_t)(x.term[e] & 1u) << 30) | ((uint32_t)(x.trunc[e] & 1u) << 31);
  }
  if (x.done != nullptr) {
    const bool vec = ((reinterpret_cast<uintptr_t>(x.term) | reinterpret_cast<uintptr_t>(x.trunc) | reinterpret_cast<uintptr_t>(x.done)) & 3u) == 0;
    if (vec) {
      for (size_t i = tid; i < n4; i += nth)
        reinterpret_cast<uint32_t*>(x.done)[i] = (reinterpret_cast<const uint32_t*>(x.term)[i] & 0x01010101u) |
                                                 ((reinterpret_cast<const uint32_t*>(x.trunc)[i] & 0x01010101u) << 1);
    }
    for (size_t e = (vec ? (n4 << 2) : 0) + tid; e < (size_t)x.n_envs; e += nth)
      x.done[e] = (uint8_t)((x.term[e] & 1u) | ((x.trunc[e] & 1u) << 1));
  }
}

// [E*W] packed -> [E,N] uint8 / float32.  One thread per output element: writes are coalesced,
// the packed word is broadcast from L1 to the N threads that share it.
template <typename OutT>
__global__ void __launch_bounds__(256) unpack_kernel(const uint64_t* __restrict__ state, OutT* __restrict__ out,
                                                    int n_genes, int W, int64_t n_envs) {
  const int64_t total = n_envs * n_genes;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = i / n_genes;
    const int g = (int)(i - e * n_genes);
    const uint64_t w = state[e * W + (g >> 6)];
    out[i] = (OutT)((w >> (g & 63)) & 1ull);
  }
}

__global__ void __launch_bounds__(256) pack_kernel(const uint8_t* __restrict__ bits, uint64_t* __restrict__ state,
                                                  int n_genes, int W, int64_t n_envs) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_envs * W;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = i / W;
    const int w = (int)(i - e * W);
    uint64_t v = 0;
    const int g1 = min(n_genes, (w + 1) * 64);
    for (int g = w * 64; g < g1; ++g) v |= (uint64_t)(bits[e * n_genes + g] & 1u) << (g & 63);
    state[i] = v;
  }
}

template <int W>
__global__ void __launch_bounds__(256) attractor_id_kernel(const __grid_constant__ NetParams n,
                                                          const uint64_t* __restrict__ state,
                                                          int32_t* __restrict__ attr_id, int64_t n_envs) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_envs;
       e += (int64_t)gridDim.x * blockDim.x) {
    uint64_t s[W];
#pragma unroll
    for (int w = 0; w < W; ++w) s[w] = state[e * W + w];
    int found = -1;
    if (n.ahash_tags != nullptr) {
      found = attractor_of_hashed<W>(n, s);
    } else {
      for (int a = 0; a < n.n_attr && found < 0; ++a)
        if (in_attractor<W>(n.attr_offset, n.attr_care, n.attr_val, a, s)) found = a;
    }
    attr_id[e] = found;
  }
}

}  // namespace pbn
