// Philox4x32-10 (Salmon et al., SC'11), counter-based: no RNG state in HBM.
// Each round is 2 IMAD.WIDE (fma pipe) + 2 three-input XORs (one LOP3 each, alu pipe);
// the key schedule is warp-uniform and folds into immediates/uniform registers.
#pragma once
#ifndef __CUDACC_RTC__
#include <stdint.h>
#endif

namespace pbn {

struct Philox4 {
  uint32_t x, y, z, w;
};

__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                 uint32_t k0, uint32_t k1) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  constexpr uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)M0 * c0;
    const uint64_t p1 = (uint64_t)M1 * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
    k0 += W0;
    k1 += W1;
  }
  return Philox4{c0, c1, c2, c3};
}

// Same function with the key schedule precomputed (rk[2r], rk[2r+1] = round-r keys): when rk lives in
// the kernel parameter block the keys become constant-bank operands of the XORs.
__device__ __forceinline__ Philox4 philox4x32_10_rk(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                    const uint32_t (&rk)[20]) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)M0 * c0;
    const uint64_t p1 = (uint64_t)M1 * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ rk[2 * r];
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ rk[2 * r + 1];
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
  }
  return Philox4{c0, c1, c2, c3};
}

__device__ __forceinline__ Philox4 philox_stream_rk(uint64_t id, uint64_t step, uint32_t kind, uint32_t idx,
                                                    const uint32_t (&rk)[20]) {
  const uint32_t c3 = ((uint32_t)(step >> 32) & 0xFFFFu) | (kind << 28) | (idx << 16);
  return philox4x32_10_rk((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)step, c3, rk);
}

// Block i of the sliced kernels' perturbation sub-stream q (0..3).  The walk draws one word per event plus one, up to
// 8N + 1 = 769 words (193 blocks) at N = 96: blocks 64q + i for the first 64, then 256 + 192q + (i - 64), so a dense
// walk never wraps onto words it has already used.
__device__ __forceinline__ uint32_t pert_block(uint32_t q, uint32_t i) {
  return i < 64u ? 64u * q + i : 256u + 192u * q + (i - 64u);
}

// Counter layout shared by every stream of the library (include/pbn_b200.h "Random streams").
__device__ __forceinline__ Philox4 philox_stream(uint64_t id, uint64_t step, uint32_t kind, uint32_t idx,
                                                 uint32_t k0, uint32_t k1) {
  const uint32_t c3 = ((uint32_t)(step >> 32) & 0xFFFFu) | (kind << 28) | (idx << 16);
  return philox4x32_10((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)step, c3, k0, k1);
}

// Selection planes of a slot with arbitrary predictor probabilities (e.g. ASSA-format PBNs, train_assa_matlab_BQN.py:
// 72-171): per env a 32-bit uniform u is compared with the gene's K-1 cumulative thresholds, sel = #{k : cum[k] <= u}
// -- the same rule, with the same 32-bit thresholds, as the thread-per-env kernel.  Bit-sliced: u's bit 31 - j of the
// column's 32 envs is plane j = word j of the slot's blocks (SELECT, 128 + 8 r + i), compared bit-serially from the
// most significant bit; planes are drawn four at a time only while some env of the warp is still undecided against
// some threshold (2^-j of them after j planes: four blocks in the typical case).  Returns lo + 2 hi = sel.
__device__ __forceinline__ void draw_weighted(uint64_t gid, uint64_t step, const uint32_t (&rk)[20], uint32_t r, uint32_t K,
                                              const uint32_t* cum, uint32_t& lo, uint32_t& hi) {
  const uint32_t c0 = cum[0], c1 = cum[1], c2 = cum[2];
  uint32_t eq0 = 0xFFFFFFFFu, eq1 = K > 2u ? 0xFFFFFFFFu : 0u, eq2 = K > 3u ? 0xFFFFFFFFu : 0u;   // still equal to the threshold
  uint32_t lt0 = 0u, lt1 = K > 2u ? 0u : 0xFFFFFFFFu, lt2 = K > 3u ? 0u : 0xFFFFFFFFu;             // decided: u < threshold
#pragma unroll 1
  for (uint32_t i = 0; i < 8u; ++i) {
    const Philox4 P = philox_stream_rk(gid, step, PBN_RNG_SELECT, 128u + 8u * r + i, rk);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t u = j == 0 ? P.x : j == 1 ? P.y : j == 2 ? P.z : P.w;
      const uint32_t sh = 4u * i + (uint32_t)j;
      const uint32_t b0 = (uint32_t)((int32_t)(c0 << sh) >> 31), b1 = (uint32_t)((int32_t)(c1 << sh) >> 31), b2 = (uint32_t)((int32_t)(c2 << sh) >> 31);
      lt0 |= eq0 & ~u & b0; eq0 &= ~(u ^ b0);
      lt1 |= eq1 & ~u & b1; eq1 &= ~(u ^ b1);
      lt2 |= eq2 & ~u & b2; eq2 &= ~(u ^ b2);
    }
    if (!__any_sync(0xFFFFFFFFu, (eq0 | eq1 | eq2) != 0u)) break;
  }
  const uint32_t g0 = ~lt0, g1 = ~lt1, g2 = ~lt2;   // u >= threshold (thermometer: g0 >= g1 >= g2)
  lo = g0 ^ g1 ^ g2;
  hi = g1;
}

// The same draw for genes with up to 8 predictors (networks with such a gene carry three selection planes,
// PBN_SELBITS == 3): up to 7 thresholds, sel = lo + 2 hi + 4 h2.  For K <= 4 it returns what draw_weighted returns.
__device__ __forceinline__ void draw_weighted8(uint64_t gid, uint64_t step, const uint32_t (&rk)[20], uint32_t r, uint32_t K,
                                               const uint32_t* cum, uint32_t& lo, uint32_t& hi, uint32_t& h2) {
  uint32_t c[7], eq[7], lt[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    c[k] = cum[k];
    const bool active = (uint32_t)k + 1u < K;
    eq[k] = active ? 0xFFFFFFFFu : 0u;   // still equal to the threshold
    lt[k] = active ? 0u : 0xFFFFFFFFu;   // decided: u < threshold
  }
#pragma unroll 1
  for (uint32_t i = 0; i < 8u; ++i) {
    const Philox4 P = philox_stream_rk(gid, step, PBN_RNG_SELECT, 128u + 8u * r + i, rk);
    uint32_t open = 0u;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t u = j == 0 ? P.x : j == 1 ? P.y : j == 2 ? P.z : P.w;
      const uint32_t sh = 4u * i + (uint32_t)j;
#pragma unroll
      for (int k = 0; k < 7; ++k) {
        const uint32_t b = (uint32_t)((int32_t)(c[k] << sh) >> 31);
        lt[k] |= eq[k] & ~u & b;
        eq[k] &= ~(u ^ b);
      }
    }
#pragma unroll
    for (int k = 0; k < 7; ++k) open |= eq[k];
    if (!__any_sync(0xFFFFFFFFu, open != 0u)) break;
  }
  // thermometer code (g0 >= g1 >= ... >= g6, g_k = u >= threshold k) -> binary
  const uint32_t g0 = ~lt[0], g1 = ~lt[1], g2 = ~lt[2], g3 = ~lt[3], g4 = ~lt[4], g5 = ~lt[5], g6 = ~lt[6];
  h2 = g3;
  hi = (g1 & ~g3) | g5;
  lo = (g0 & ~g1) | (g2 & ~g3) | (g4 & ~g5) | g6;
}

}  // namespace pbn
