// Exact finite-horizon control (include/pbn_b200.h, "Exact optimal control"): the two device operators of one
// backward-induction backup over all 2^N states of a network with N <= PBN_DP_MAX_GENES genes.
//   expect : w = P u, P = one step of the handle's dynamics without interventions (selection, then perturbation)
//   improve: v[s] = max over flip masks m of fl(r_action * |m|) + w[s ^ m], policy[s] = the maximising m
// and the forward operator of expect, for state distributions:
//   push   : y = x P (x P_mu with interventions), the same successor enumeration as a fixed-point scatter
// Generic kernels over the handle's NetParams (like discover.cuh): states are one 32-bit index (bit i = gene i),
// every launch covers a bounded slice of the state space, and no floating-point sum uses atomics (push adds integers),
// so the results are bit-identical from call to call.
#pragma once
#include "pbn_common.cuh"
#include "discover.cuh"

namespace pbn {

constexpr int kDpWarps = 8;          // warps per CTA of the expect kernel
constexpr int kDpChunks = 6;         // free genes beyond the 5 lane genes, in digits of 4 bits: 5 + 6 * 4 >= 28
constexpr int kKpTileBits = 10;      // the low genes of the perturbation channel, folded in one shared-memory pass

// ---- expect: (F u)(x) = sum over the successor set of x of prod_i (q_i or 1 - q_i) * u[t] -------------------------
// One warp per state.  Lane g < N evaluates gene g's predictors (eval_func, shared with the successor descriptor) and
// forms q1 = sum of the selection probabilities of the predictors that yield 1, q0 = of those that yield 0; two ballots
// give the fixed genes and the free ones (q1 > 0 and q0 > 0 as sets: some predictor yields each value).  The lowest
// min(free, 5) free genes are spread over the lanes (lane l takes their assignment l); the remaining free genes are
// enumerated by every lane in digits of 4 genes whose weight products and bit patterns sit in per-warp tables.  The sum
// runs in a fixed order (inner digit innermost, then the other digits, then a shuffle tree over the lanes), so it is
// deterministic.
struct ExpectWarpTables {
  double wt[kDpChunks][16];
  uint32_t bits[kDpChunks][16];
};

__global__ void __launch_bounds__(kDpWarps * 32) dp_expect_kernel(const __grid_constant__ NetParams n,
                                                                 const double* __restrict__ func_prob,
                                                                 const double* __restrict__ src, double* __restrict__ w,
                                                                 uint32_t s0, uint32_t count) {
  __shared__ ExpectWarpTables tabs[kDpWarps];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  ExpectWarpTables& tb = tabs[warp];
  for (uint32_t i = blockIdx.x * kDpWarps + warp; i < count; i += gridDim.x * kDpWarps) {
    const uint32_t x = s0 + i;
    double q1 = 0.0, q0 = 0.0;
    bool can1 = false, can0 = false;
    if ((int)lane < n.n_genes) {
      const uint64_t s[1] = {x};
      for (int f = n.func_offset[lane]; f < n.func_offset[lane + 1]; ++f) {
        const double p = func_prob[f];
        if (eval_func<1>(n, f, s)) { q1 += p; can1 = true; } else { q0 += p; can0 = true; }
      }
    }
    const uint32_t one = __ballot_sync(0xFFFFFFFFu, can1), zero = __ballot_sync(0xFFFFFFFFu, can0);
    uint32_t fr = one & zero;
    const uint32_t fixed = one & ~zero;
    const int nf = __popc(fr);
    const int nlo = nf < 5 ? nf : 5;
    // lane part: the lowest nlo free genes
    double wlo = 1.0;
    uint32_t tlo = 0;
    for (int j = 0; j < nlo; ++j) {
      const int g = __ffs(fr) - 1;
      fr &= fr - 1;
      const double a1 = __shfl_sync(0xFFFFFFFFu, q1, g), a0 = __shfl_sync(0xFFFFFFFFu, q0, g);
      const bool b = (lane >> j) & 1u;
      wlo *= b ? a1 : a0;
      tlo |= (uint32_t)b << g;
    }
    // digit tables of the remaining free genes: digit k holds genes 4k..4k+3 of them
    const int nhi = nf - nlo;
    double dw = 1.0;
    uint32_t db = 0;
    for (int j = 0; j < nhi; ++j) {
      const int g = __ffs(fr) - 1;
      fr &= fr - 1;
      const double a1 = __shfl_sync(0xFFFFFFFFu, q1, g), a0 = __shfl_sync(0xFFFFFFFFu, q0, g);
      const bool b = (lane >> (j & 3)) & 1u;
      dw *= b ? a1 : a0;
      db |= (uint32_t)b << g;
      if ((j & 3) == 3 || j == nhi - 1) {
        if (lane < 16u) { tb.wt[j >> 2][lane] = dw; tb.bits[j >> 2][lane] = db; }
        dw = 1.0;
        db = 0;
      }
    }
    __syncwarp();
    double acc = 0.0;
    if (lane < (1u << nlo)) {
      const int b0 = nhi < 4 ? nhi : 4;
      const int nd = (nhi + 3) >> 2;                // digits in use (the first one is the inner loop)
      const uint32_t outer = 1u << (nhi - b0), inner = 1u << b0;
      const uint32_t base = fixed | tlo;
      for (uint32_t xo = 0; xo < outer; ++xo) {
        double wo = wlo;
        uint32_t to = base;
        uint32_t r = xo;
        for (int k = 1; k < nd; ++k) {
          wo *= tb.wt[k][r & 15u];
          to |= tb.bits[k][r & 15u];
          r >>= 4;
        }
        double sum = 0.0;
        if (nhi == 0) {
          sum = src[to];
        } else {
#pragma unroll 4
          for (uint32_t x0 = 0; x0 < inner; ++x0) sum += tb.wt[0][x0] * src[to | tb.bits[0][x0]];
        }
        acc += wo * sum;
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_down_sync(0xFFFFFFFFu, acc, off);
    if (lane == 0) w[x] = acc;
    __syncwarp();   // the tables are rewritten for the next state
  }
}

// ---- the binary symmetric perturbation channel K_p = (x)_i [[1-p, p], [p, 1-p]] ------------------------------------
// Low genes: one CTA per tile of 2^tb consecutive states runs the butterflies of genes 0..tb-1 in shared memory.
__global__ void __launch_bounds__(256) dp_kp_low_kernel(const double* __restrict__ in, double* __restrict__ out, int tb,
                                                        uint32_t tile0, uint32_t n_tiles, double p) {
  __shared__ double sm[1 << kKpTileBits];
  const uint32_t size = 1u << tb;
  const double q = 1.0 - p;
  for (uint32_t t = tile0 + blockIdx.x; t < tile0 + n_tiles; t += gridDim.x) {
    const size_t base = (size_t)t << tb;
    for (uint32_t j = threadIdx.x; j < size; j += blockDim.x) sm[j] = in[base + j];
    for (int b = 0; b < tb; ++b) {
      __syncthreads();
      for (uint32_t j = threadIdx.x; j < (size >> 1); j += blockDim.x) {
        const uint32_t lo = ((j >> b) << (b + 1)) | (j & ((1u << b) - 1u)), hi = lo | (1u << b);
        const double a = sm[lo], z = sm[hi];
        sm[lo] = q * a + p * z;
        sm[hi] = q * z + p * a;
      }
    }
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < size; j += blockDim.x) out[base + j] = sm[j];
    __syncthreads();
  }
}

// One higher gene b, in place: pairs (x, x ^ 2^b) with bit b of x clear, pair index j in [j0, j0 + count).
__global__ void __launch_bounds__(256) dp_kp_bit_kernel(double* __restrict__ v, int b, uint32_t j0, uint32_t count, double p) {
  const double q = 1.0 - p;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const uint32_t j = j0 + i;
    const uint32_t lo = ((j >> b) << (b + 1)) | (j & ((1u << b) - 1u)), hi = lo | (1u << b);
    const double a = v[lo], z = v[hi];
    v[lo] = q * a + p * z;
    v[hi] = q * z + p * a;
  }
}

// Perturbation model A: w = c * (F u) + K_p u - c * u with c = (1 - p)^N (w holds F u on entry).
__global__ void __launch_bounds__(256) dp_mix_kernel(double* __restrict__ w, const double* __restrict__ kpu,
                                                     const double* __restrict__ u, double c, uint32_t s0, uint32_t count) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const uint32_t x = s0 + i;
    w[x] = (c * w[x] + kpu[x]) - c * u[x];
  }
}

// ---- push: y = x F, the transpose of expect -------------------------------------------------------------------------
// A scatter, made deterministic by fixed point: every term x[s] F(s -> t) is rounded to the nearest multiple of 2^-63
// and added to y[t] as an unsigned 64-bit integer.  Integer addition is associative, so the sum does not depend on the
// order in which the atomics land; dp_fix_kernel converts each total to fp64 once.  For x >= 0 with sum x <= 1 the
// totals stay below 2^64 units.  A term loses at most 2^-64 to the rounding (terms below 2^-64 vanish).
constexpr double kDpFixOne = 9223372036854775808.0;   // 2^63: fixed-point units per 1.0

__device__ __forceinline__ void dp_fix_add(unsigned long long* __restrict__ acc, uint32_t t, double v) {
  const unsigned long long q = __double2ull_rn(v * kDpFixOne);
  if (q != 0ull) atomicAdd(acc + t, q);
}

// One warp per source state s, enumerating its successors with dp_expect_kernel's code (lane genes, ballots, digit
// tables; repeated here so that expect compiles as before); each term x[s] * weight is added to y[t] instead of
// gathering u[t].  A state with x[s] = 0 is skipped, so a push from a point mass or a sparse distribution costs one pass
// over x plus its terms.
__global__ void __launch_bounds__(kDpWarps * 32) dp_push_kernel(const __grid_constant__ NetParams n,
                                                               const double* __restrict__ func_prob,
                                                               const double* __restrict__ x,
                                                               unsigned long long* __restrict__ y, uint32_t s0,
                                                               uint32_t count) {
  __shared__ ExpectWarpTables tabs[kDpWarps];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  ExpectWarpTables& tb = tabs[warp];
  for (uint32_t i = blockIdx.x * kDpWarps + warp; i < count; i += gridDim.x * kDpWarps) {
    const uint32_t s = s0 + i;
    const double xs = x[s];
    if (xs == 0.0) continue;   // the same for every lane of the warp
    double q1 = 0.0, q0 = 0.0;
    bool can1 = false, can0 = false;
    if ((int)lane < n.n_genes) {
      const uint64_t st[1] = {s};
      for (int f = n.func_offset[lane]; f < n.func_offset[lane + 1]; ++f) {
        const double p = func_prob[f];
        if (eval_func<1>(n, f, st)) { q1 += p; can1 = true; } else { q0 += p; can0 = true; }
      }
    }
    const uint32_t one = __ballot_sync(0xFFFFFFFFu, can1), zero = __ballot_sync(0xFFFFFFFFu, can0);
    uint32_t fr = one & zero;
    const uint32_t fixed = one & ~zero;
    const int nf = __popc(fr);
    const int nlo = nf < 5 ? nf : 5;
    // lane part: the lowest nlo free genes
    double wlo = 1.0;
    uint32_t tlo = 0;
    for (int j = 0; j < nlo; ++j) {
      const int g = __ffs(fr) - 1;
      fr &= fr - 1;
      const double a1 = __shfl_sync(0xFFFFFFFFu, q1, g), a0 = __shfl_sync(0xFFFFFFFFu, q0, g);
      const bool b = (lane >> j) & 1u;
      wlo *= b ? a1 : a0;
      tlo |= (uint32_t)b << g;
    }
    // digit tables of the remaining free genes: digit k holds genes 4k..4k+3 of them
    const int nhi = nf - nlo;
    double dw = 1.0;
    uint32_t db = 0;
    for (int j = 0; j < nhi; ++j) {
      const int g = __ffs(fr) - 1;
      fr &= fr - 1;
      const double a1 = __shfl_sync(0xFFFFFFFFu, q1, g), a0 = __shfl_sync(0xFFFFFFFFu, q0, g);
      const bool b = (lane >> (j & 3)) & 1u;
      dw *= b ? a1 : a0;
      db |= (uint32_t)b << g;
      if ((j & 3) == 3 || j == nhi - 1) {
        if (lane < 16u) { tb.wt[j >> 2][lane] = dw; tb.bits[j >> 2][lane] = db; }
        dw = 1.0;
        db = 0;
      }
    }
    __syncwarp();
    if (lane < (1u << nlo)) {
      const int b0 = nhi < 4 ? nhi : 4;
      const int nd = (nhi + 3) >> 2;
      const uint32_t outer = 1u << (nhi - b0), inner = 1u << b0;
      const uint32_t base = fixed | tlo;
      for (uint32_t xo = 0; xo < outer; ++xo) {
        double wo = xs * wlo;
        uint32_t to = base;
        uint32_t r = xo;
        for (int k = 1; k < nd; ++k) {
          wo *= tb.wt[k][r & 15u];
          to |= tb.bits[k][r & 15u];
          r >>= 4;
        }
        if (nhi == 0) {
          dp_fix_add(y, to, wo);
        } else {
#pragma unroll 4
          for (uint32_t x0 = 0; x0 < inner; ++x0) dp_fix_add(y, to | tb.bits[0][x0], wo * tb.wt[0][x0]);
        }
      }
    }
    __syncwarp();   // the tables are rewritten for the next state
  }
}

// The interventions of a closed loop, y = x M_mu: x[s] moves to s ^ masks[s] (mask bits at gene N and above, outside
// smask = 2^N - 1, are ignored), into the same fixed-point accumulator.
__global__ void __launch_bounds__(256) dp_flip_push_kernel(const double* __restrict__ x, const uint32_t* __restrict__ masks,
                                                           unsigned long long* __restrict__ y, uint32_t smask, uint32_t s0,
                                                           uint32_t count) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const uint32_t s = s0 + i;
    const double xs = x[s];
    if (xs != 0.0) dp_fix_add(y, (s ^ masks[s]) & smask, xs);
  }
}

// Fixed point to fp64 in place: v[s] = units * 2^-63.
__global__ void __launch_bounds__(256) dp_fix_kernel(unsigned long long* __restrict__ v, uint32_t s0, uint32_t count) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const uint32_t s = s0 + i;
    v[s] = (unsigned long long)__double_as_longlong(__ull2double_rn(v[s]) * (1.0 / kDpFixOne));
  }
}

// ---- improve: ball relaxation ---------------------------------------------------------------------------------------
// B_0(s) = (w[s], s); B_k(s) = best(B_{k-1}(s), best over i in G of B_{k-1}(s ^ e_i)), best = larger value, then smaller
// endpoint: B_k(s) is the best endpoint within k flips of G.  Pass k (k = 1..max_flips) reads B_{k-1} (bval/bend, or w
// with endpoint = index for k = 1), writes B_k (unless it is the last pass) and offers the candidate
// fl(r_action * k) + B_k.value to (v, policy); a candidate replaces the incumbent only when strictly larger, so the
// fewest flips win ties.  Pass 0 (max_flips = 0) writes v = fl(r_action * 0) + w, policy = 0.
__device__ __forceinline__ bool dp_better(double va, uint32_t ea, double vb, uint32_t eb) {
  return va > vb || (va == vb && ea < eb);
}

__global__ void __launch_bounds__(256) dp_improve_kernel(const double* __restrict__ w, const double* __restrict__ bval,
                                                         const uint32_t* __restrict__ bend, double* __restrict__ oval,
                                                         uint32_t* __restrict__ oend, double* __restrict__ v,
                                                         uint32_t* __restrict__ policy, uint32_t genes, int k,
                                                         double cost0, double cost_k, uint32_t s0, uint32_t count) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const uint32_t s = s0 + i;
    double vin;
    uint32_t pin;
    if (k <= 1) {
      vin = __dadd_rn(cost0, w[s]);
      pin = 0u;
      if (k == 0) {
        v[s] = vin;
        if (policy != nullptr) policy[s] = 0u;
        continue;
      }
    } else {
      vin = v[s];
      pin = policy != nullptr ? policy[s] : 0u;
    }
    double bv;
    uint32_t be;
    if (bend == nullptr) { bv = w[s]; be = s; } else { bv = bval[s]; be = bend[s]; }
    uint32_t g = genes;
    while (g) {
      const uint32_t t = s ^ (g & (0u - g));
      g &= g - 1u;
      double cv;
      uint32_t ce;
      if (bend == nullptr) { cv = w[t]; ce = t; } else { cv = bval[t]; ce = bend[t]; }
      if (dp_better(cv, ce, bv, be)) { bv = cv; be = ce; }
    }
    if (oend != nullptr) { oval[s] = bv; oend[s] = be; }
    const double cand = __dadd_rn(cost_k, bv);
    if (cand > vin) { vin = cand; pin = s ^ be; }
    v[s] = vin;
    if (policy != nullptr) policy[s] = pin;
  }
}

}  // namespace pbn
