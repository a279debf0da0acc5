// Bit-sliced step kernel: the fast path, specialised per network at load time (NVRTC).
//
// Layout of the work
//   A CTA of 4 warps owns a tile of 1024 consecutive env instances.  "Column" L (= lane id, in
//   every warp) owns the 32 envs
//       env(L, j, c) = tile_base + 128*j + 4*L + c,   j = 0..7, c = 0..3,   slice bit b = 4*j + c
//   so every global access is a coalesced vector access (4 consecutive envs per lane: 32 B of
//   state, 4*BINS action bytes, 16 B of target ids / rewards, 8 B of step counters, 4 B of flags).
//   The column's 32 packed states are transposed into N bit-planes (plane i, bit b = gene i of
//   env b): from then on one 32-bit logic instruction advances 32 envs at once.
//
//   The four warps split every phase of the tile (all exchange goes through shared memory, each
//   thread only ever touches its own column; three block barriers per tile):
//     A  warp w loads groups j = 2w, 2w+1 (8 envs per lane), applies the interventions, keeps the
//        s1 rows in registers and publishes them                                   -> S1 rows
//     B  warp w gathers byte w of all 32 rows and finishes an 8x8-block bit transpose
//        = planes 8w..8w+7 of each 32-gene word                                    -> PL planes
//     C1 warp w draws the selection planes of slots r = w, w+4, ... from Philox   -> SEL planes
//     C2 warp w evaluates "its" genes: generated LOP3 trees (net_update.inc)       -> OPL planes
//     E  warp w gathers byte w of all out planes, 8x8-block transpose = its 8 next-state rows
//     D  sparse perturbation events of the column, applied by the warp that owns the row
//     F  target test, counters, reward, vector stores for its 8 envs; G auto-reset
//
// Code shape (profiles/r01_notes.md): a first, fully unrolled one-warp-per-tile version of this
// kernel starved for instructions (300 KB of straight-line SASS); a compact-loop one-warp version
// was latency-bound (1.7 warps per scheduler at 2^20 envs).  Hence four warps per tile, and only
// the predictor functions themselves (LOP3 trees whose immediates are the truth tables) are
// generated straight-line code.
//
// Random streams (DESIGN.md "Sliced random stream"; CPU twin: oracle/pbn_oracle.py sliced_stream)
//   group id = (env >> 10) * 32 + ((env >> 2) & 31)  (= tile * 32 + lane), slice bit as above.
//   SELECT: the genes with K > 1 predictors get slots r = 0, 1, ... in gene order; slot r owns Philox block
//           (SELECT, r) = words x, y, z, w.  K=2 uses x (s0), K=4 x, y (s0, s1), K=3 the pairs (x, y), (z, w): pair
//           value 3 is rejected and replaced by the next pair.  The 1/16 of the positions still at 3 are settled by
//           the pool of the slot's group q = r mod 4: Philox blocks (FIX, 1024 q + i), i = 0, 1, ...; each block is two
//           pair-planes (x, y), (z, w); per pair-plane the group's K=3 slots r = q, q + 4, ... in that order take
//           bit b of the plane if they are still at 3 there and no earlier slot of the group has claimed bit b of this
//           plane; blocks are consumed until no slot of the group is at 3 anywhere in the column.  Exactly uniform
//           1-of-3, all choices independent (no random pair is used twice).  sel = s0 + 2*s1.
//   PERTURB: sub-stream q = b >> 3 (Philox blocks (PERTURB, 64q + i)) covers the 8 slice bits
//           8q..8q+7: geometric skipping over slots gene*8 + (b & 7) with survival table S[0..8N].
//   RESET:  per env (global env id), as in the scalar kernel.
//
// Algorithmic HBM bytes per env-step: 33 (N <= 64) / 49 (N <= 128), see step_scalar.cuh.
#pragma once
#include "pbn_common.cuh"

#ifndef PBN_N
#error "net_gen.cuh must be included first"
#endif

namespace pbn {

#define PBN_RNG_FIX 3u

constexpr int kSlots = 8 * PBN_N;             // perturbation slots per (column, warp) sub-stream
constexpr int kNW = PBN_NW32;                 // 32-bit words per state
constexpr int kW64 = (PBN_N <= 64) ? 1 : 2;   // 64-bit words per state in HBM
constexpr uint32_t kLastMask = (PBN_N % 32) ? ((1u << (PBN_N % 32)) - 1u) : 0xFFFFFFFFu;
constexpr int kWarps = 4;                     // warps per tile (PBN_THREADS == 128)

// per-CTA scratch, in 32-bit words; every array is [row][lane]
constexpr int kScrRows = 0;                          // s1 rows                      [kNW*32][32]
constexpr int kScrPl = kScrRows + kNW * 32 * 32;     // PL input planes              [kNW*32][32]
constexpr int kScrSel0 = kScrPl + kNW * 32 * 32;     // selection planes s0          [PBN_NSEL][32]
constexpr int kScrSel1 = kScrSel0 + PBN_NSEL * 32;   // selection planes s1          [PBN_NSEL][32]
// (PBN_SELBITS == 3, networks with a gene of 5..8 predictors: a third plane set s2 follows s1 -- sel1 + PBN_NSEL * 32)
constexpr int kScrStat = kScrSel1 + (PBN_SELBITS - 1) * PBN_NSEL * 32;   // 8 block-level statistics counters
constexpr int kEvWords = (8 * PBN_N < 255) ? 1 : 2;  // packed words of pre-drawn perturbation events per thread
constexpr int kScrEv = kScrStat + 8;                 // pre-drawn perturbation events              [kEvWords][128]
constexpr int kScrPm = kScrEv + 128 * kEvWords;      // model A: envs with a perturbation event, byte w of word [lane] = rows 8w..8w+7
constexpr int kScrWords = kScrPm + 32;               // total (must equal PBN_SCRATCH_WORDS)
// Pre-drawn perturbation events of a thread: ascending slot positions, kEvBits each, packed into kEvWords words;
// all-ones = no event; an all-zero first word (never a valid ascending list) = more than kEvCap events: phase D
// redoes the walk.
constexpr uint32_t kEvBits = (kSlots < 255) ? 8u : 10u;
constexpr uint32_t kEvPerWord = 32u / kEvBits;
constexpr uint32_t kEvCap = kEvPerWord * kEvWords;   // 4 events for N <= 31, else 6
constexpr uint32_t kEvMask = (1u << kEvBits) - 1u;
constexpr uint32_t kPreEvOverflow = 0u;
static_assert(kSlots < (int)kEvMask, "pre-drawn event positions do not fit their field");
#if PBN_SELBITS == 3
#define PBN_SEL2_OF(sel1) (sel1) + PBN_NSEL * 32,
#else
#define PBN_SEL2_OF(sel1)
#endif
static_assert(kScrWords == PBN_SCRATCH_WORDS, "host and device disagree on the scratch size");
static_assert(PBN_THREADS == 32 * kWarps, "one tile per 4-warp CTA");

__device__ __forceinline__ uint32_t shl_clamp(uint32_t v, uint32_t s) {
  uint32_t r;
  asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(s));  // shift counts > 31 give 0
  return r;
}

template <int IMM>
__device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(r) : "r"(a), "r"(b), "r"(c), "n"(IMM));
  return r;
}

// a ? b : c, bitwise
__device__ __forceinline__ uint32_t bmux(uint32_t a, uint32_t b, uint32_t c) { return lop3<0xCA>(a, b, c); }

// One quarter of a 32x32 bit transpose.  `src` is a [32][32-lane] scratch array holding the 32 source
// rows of this column; the result is rows 8q..8q+7 of the transposed matrix: out[i] bit b = (source
// row b) bit 8q+i.  The two byte-granular butterfly stages are the byte gather below (byte q of rows
// i, i+8, i+16, i+24), the three bit-granular ones run on the 8 registers.
__device__ __forceinline__ void transpose_quarter(const uint32_t* src, uint32_t q, uint32_t (&out)[8]) {
  const uint8_t* sb = reinterpret_cast<const uint8_t*>(src) + q;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint32_t b0 = sb[(i)*128], b1 = sb[(i + 8) * 128], b2 = sb[(i + 16) * 128], b3 = sb[(i + 24) * 128];
    out[i] = __byte_perm(__byte_perm(b0, b1, 0x0040), __byte_perm(b2, b3, 0x0040), 0x5410);
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint32_t lo = out[k], hi = out[k + 4];
    out[k] = bmux(0x0F0F0F0Fu, lo, hi << 4);
    out[k + 4] = bmux(0x0F0F0F0Fu, lo >> 4, hi);
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    if (k & 2) continue;
    const uint32_t lo = out[k], hi = out[k + 2];
    out[k] = bmux(0x33333333u, lo, hi << 2);
    out[k + 2] = bmux(0x33333333u, lo >> 2, hi);
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    if (k & 1) continue;
    const uint32_t lo = out[k], hi = out[k + 1];
    out[k] = bmux(0x55555555u, lo, hi << 1);
    out[k + 1] = bmux(0x55555555u, lo >> 1, hi);
  }
}

// ---- TMA (1-D bulk copy) staging of a tile's state and action bytes into shared memory -------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// Warm the L2 with a range that will be bulk-copied once the previous launch has completed (coherent: lines
// the previous launch still writes are simply updated in place).
__device__ __forceinline__ void l2_prefetch(const void* src, uint32_t bytes) {
  if ((reinterpret_cast<unsigned long long>(src) & 15ull) == 0ull)   // the bulk prefetch wants 16-byte aligned ranges; it is only a hint
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "PBN_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra PBN_DONE;\n"
      "bra PBN_WAIT;\n"
      "PBN_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Development aid, compiled only into specialisations built with PBN_B200_PROFILE=1 in the environment
// (scripts/phase_probe.py): with flag bit 31 set, thread 0 of CTA 0 writes %globaltimer stamps (ns) of the phase
// boundaries into final_state[E*W .. E*W+15], and thread 0 of every CTA its start/end stamps (+ SM id in
// the top byte) into final_state[E*W + 16 + 8*blockIdx + {0,7}] (1: input copy arrived, 2: out planes done,
// 3..6: after phases E, D, F, G):
// the caller provides the extra words.
__device__ __forceinline__ void phase_stamp(const pbn_step_args& a, int i) {
#ifdef PBN_PROFILE
  if ((a.flags & 0x80000000u) && blockIdx.x == 0 && threadIdx.x == 0 && a.final_state != nullptr) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    a.final_state[a.n_envs * kW64 + i] = t;
  }
#else
  (void)a; (void)i;
#endif
}
__device__ __forceinline__ void cta_stamp(const pbn_step_args& a, int which) {
#ifdef PBN_PROFILE
  if ((a.flags & 0x80000000u) && threadIdx.x == 0 && a.final_state != nullptr) {
    unsigned long long t;
    unsigned int smid;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
    a.final_state[a.n_envs * kW64 + 16 + 8 * blockIdx.x + which] =
        (t & 0x00FFFFFFFFFFFFFFull) | ((unsigned long long)smid << 56);
  }
#else
  (void)a; (void)which;
#endif
}

__device__ __forceinline__ uint32_t pick4(const Philox4& b, uint32_t q) {
  return q == 0 ? b.x : q == 1 ? b.y : q == 2 ? b.z : b.w;
}

// Survival table S[j] = floor((1-p)^j 2^32), j = 0..8N, of the perturbation sub-streams: filled per handle after
// the library is loaded (constant memory: the look-ups of the geometric skip are data-dependent and
// lane-divergent; from global memory each step of the search cost a DRAM/L2 round trip, ~2 us per event).
__constant__ uint32_t kSurvTable[kSlots + 1];

// Next event distance of the perturbation stream: 1 + max{j in 0..8N : u < S[j]} (S[0] = 2^32 conceptually).
// S is geometric, so j is first guessed as log2(u / 2^32) / log2(1 - p) and pinned down exactly by four
// INDEPENDENT table reads around the guess (one memory latency instead of a dependent binary search, whose
// steps are lane-divergent); if the window misses (tiny p, float error) the binary search decides.
__device__ __noinline__ int pert_search(const NetParams& n, uint32_t u) {
  const uint32_t* __restrict__ S = n.surv_sliced;
  int j0 = (int)((__log2f((float)u + 1.0f) - 32.0f) * n.pert_inv_log2);
  j0 = min(max(j0, 1), kSlots);
  const int ja = j0 - 1, jd = j0 + 2;
  const bool ca = ja < 1 || u < __ldg(S + min(max(ja, 1), kSlots));
  const bool cb = u < __ldg(S + j0);
  const bool cc = j0 + 1 <= kSlots && u < __ldg(S + min(j0 + 1, kSlots));
  const bool cd = jd <= kSlots && u < __ldg(S + min(jd, kSlots));
  if (ca && !cd) return ja + (cb ? 1 : 0) + (cc ? 1 : 0) + 1;   // c(j) = (u < S[j]) is non-increasing in j
  int lo = 0, hi = kSlots;  // invariant: u < S[lo]
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (u < kSurvTable[mid]) lo = mid; else hi = mid - 1;
  }
  return lo + 1;
}

}  // namespace pbn

#include "net_update.inc"  // generated: kSelGene[], kSelK[], pbn::pbn_update_part(w, PL, OPL, SEL0, SEL1)

namespace pbn {

#if !PBN_INJECTED
// Perturbation events of this thread's (column, warp) sub-stream for one step.  They depend only on
// (column id, step counter, seed), so they are drawn early -- under the previous kernel's tail with
// programmatic dependent launch, else behind the tile's TMA copy -- and phase D only applies them: the
// Philox block and the dependent table look-ups of the geometric skip are a pure latency chain
// (≈2 us per tile when it sat in D).  One packed word per thread (see kEvBits).
// rows8 (step kernel, perturbation model A): receives the 8-bit mask of this thread's rows with at least one event --
// complete even when the packed list overflows (the walk then goes on for the mask alone).
__device__ __forceinline__ void draw_pert_events(const NetParams& n, uint32_t* ev, uint64_t gid, uint64_t step_ctr, uint32_t w,
                                                 unsigned char* rows8 = nullptr) {
  uint32_t word[kEvWords];
#pragma unroll
  for (int q = 0; q < kEvWords; ++q) word[q] = 0xFFFFFFFFu;   // no event
  uint32_t m8 = 0u;
  if (n.pert_rng && n.pert_mode != PBN_PERT_NONE) {
    const bool whole_walk = rows8 != nullptr && n.pert_mode == PBN_PERT_A;
    // none is left in the rem slots after pos iff u < S[rem]: one table read settles the usual case, the search runs
    // for real events only
    uint32_t s_rem = kSurvTable[kSlots];
    Philox4 blk = philox_stream_rk(gid, step_ctr, PBN_RNG_PERTURB, 64u * w, n.rk);
    int pos = -1;
#pragma unroll 1
    for (uint32_t k = 0;; ++k) {   // up to kEvCap events are packed
      if (k != 0u && (k & 3u) == 0u) blk = philox_stream_rk(gid, step_ctr, PBN_RNG_PERTURB, 64u * w + ((k >> 2) & 63u), n.rk);   // rare
      const uint32_t u = pick4(blk, k & 3u);
      if (u < s_rem) break;
      pos += pert_search(n, u);
      if (pos >= kSlots) break;
      s_rem = __ldg(n.surv_sliced + (kSlots - 1 - pos));
      m8 |= 1u << ((uint32_t)pos & 7u);
      if (k < kEvCap) {
        const uint32_t sh = kEvBits * (k % kEvPerWord);
#pragma unroll
        for (int q = 0; q < kEvWords; ++q)
          if ((uint32_t)q == k / kEvPerWord) word[q] = (word[q] & ~(kEvMask << sh)) | ((uint32_t)pos << sh);
      } else {
        word[0] = kPreEvOverflow;              // more than kEvCap events: the consumer redoes the walk
        if (!whole_walk) break;
      }
    }
  }
  if (rows8 != nullptr) *rows8 = (unsigned char)m8;
#pragma unroll
  for (int q = 0; q < kEvWords; ++q) ev[128 * q] = word[q];
}
#endif

// Stage the small read-only tables into shared memory (first tile of a CTA, after its global loads
// were issued; everything staged here is first read after block barrier (1)).
template <bool ASMEM>
__device__ __forceinline__ void stage_tables(const NetParams& n, const SlicedSmemLayout& L, uint32_t* s_surv,
                                             float* s_rew, int32_t* s_aoffs, uint32_t* s_aent, uint32_t* s_stat) {
  (void)s_surv;  // the survival table is read through the read-only path where needed
  if (threadIdx.x < 18) {
    const uint32_t nf = threadIdx.x % 9u;
    const bool hit = threadIdx.x >= 9;
    const float base = __fadd_rn(n.r_step, __fmul_rn(n.r_action, (float)nf));
    s_rew[threadIdx.x] = __fadd_rn(base, hit ? n.r_success : 0.0f);
  }
  if (threadIdx.x < 8) s_stat[threadIdx.x] = 0u;
  if (L.attractors_in_smem) {
    for (int i = threadIdx.x; i < n.n_attr_states * kNW; i += blockDim.x) {
      const int en = i / kNW, wd = i - en * kNW;
      s_aent[en * 2 * kNW + wd] = (uint32_t)(n.attr_care[en * kW64 + (wd >> 1)] >> (32 * (wd & 1)));
      s_aent[en * 2 * kNW + kNW + wd] = (uint32_t)(n.attr_val[en * kW64 + (wd >> 1)] >> (32 * (wd & 1)));
    }
    for (int i = threadIdx.x; i <= n.n_attr; i += blockDim.x) s_aoffs[i] = n.attr_offset[i];
  } else if (!ASMEM && L.singles_in_smem) {   // first entry + entry count of every attractor (see SlicedSmemLayout)
    for (int i = threadIdx.x; i < n.n_attr * kNW; i += blockDim.x) {
      const int at = i / kNW, wd = i - at * kNW, en = n.attr_offset[at];
      s_aent[at * 2 * kNW + wd] = (uint32_t)(n.attr_care[en * kW64 + (wd >> 1)] >> (32 * (wd & 1)));
      s_aent[at * 2 * kNW + kNW + wd] = (uint32_t)(n.attr_val[en * kW64 + (wd >> 1)] >> (32 * (wd & 1)));
    }
    for (int i = threadIdx.x; i < n.n_attr; i += blockDim.x) s_aoffs[i] = n.attr_offset[i + 1] - n.attr_offset[i];
  }
}

#if !PBN_INJECTED
// Selection planes of group w (net_update.inc: pbn_draw_group; the same streams as the plane-resident kernel) into
// the SEL scratch.  One out-of-line copy: the kernel calls it from several places.
__device__ __noinline__ void draw_group_to_scratch(const uint32_t (&rk)[20], uint32_t* sel0, uint32_t* sel1, uint64_t gid,
                                                  uint64_t step_ctr, uint32_t w) {
  uint32_t lo[PBN_MAXS4], hi[PBN_MAXS4];
#if PBN_SELBITS == 3
  uint32_t h2[PBN_MAXS4];
  pbn_draw_group(w, gid, step_ctr, rk, lo, hi, h2);
#else
  pbn_draw_group(w, gid, step_ctr, rk, lo, hi);
#endif
#pragma unroll
  for (int k = 0; k < PBN_MAXS4; ++k) {
    const int r = (int)w + 4 * k;
    if (r < PBN_NSEL) {
      sel0[r * 32] = lo[k];
      sel1[r * 32] = hi[k];
#if PBN_SELBITS == 3
      sel1[(PBN_NSEL + r) * 32] = h2[k];
#endif
    }
  }
}
#endif

// ---- C1. selection planes of this warp's slots (independent of the state) -------------------------
template <bool FULL>
__device__ __forceinline__ void draw_selection_planes(const pbn_step_args& a, const NetParams& n, uint32_t* sel0,
                                                      uint32_t* sel1, uint64_t gid, uint64_t step_ctr, int64_t e0,
                                                      uint32_t w) {
#if PBN_INJECTED
  const int64_t E = a.n_envs;
#pragma unroll 1
  for (int r = (int)w; r < PBN_NSEL; r += kWarps) {
    const uint32_t g = kSelGene[r], K = kSelK[r];
    uint32_t s0 = 0u, s1 = 0u, s2 = 0u;
    for (int b = 0; b < 32; ++b) {
      const int64_t env = e0 + 128 * (b >> 2) + (b & 3);
      uint32_t v = (env < E) ? a.sel[env * PBN_N + g] : 0u;
      v = v < K ? v : K - 1u;
      s0 |= (v & 1u) << b;
      s1 |= ((v >> 1) & 1u) << b;
      s2 |= ((v >> 2) & 1u) << b;
    }
    sel0[r * 32] = s0;
    sel1[r * 32] = s1;
#if PBN_SELBITS == 3
    sel1[(PBN_NSEL + r) * 32] = s2;
#else
    (void)s2;
#endif
  }
#else
  draw_group_to_scratch(n.rk, sel0, sel1, gid, step_ctr, w);
#endif
}

// The uncommon membership tests of phase F, out of line so that they cost the common path neither registers nor
// instruction-cache space: state in attractor a through the hash set (large attractors) or by the scan over the table
// in global memory (bit 0 of the result), and, with r_wrong != 0, state in an attractor OTHER than a (bit 1).
// (the row travels by value: a reference would force the caller's row registers into local memory)
__device__ __noinline__ uint32_t rare_membership(const NetParams& n, int a, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
  const uint32_t row[4] = {r0, r1, r2, r3};
  uint64_t y64[kW64];
#pragma unroll
  for (int wd = 0; wd < kW64; ++wd)
    y64[wd] = ((uint64_t)((2 * wd + 1 < kNW) ? row[(2 * wd + 1 < kNW) ? 2 * wd + 1 : 0] : 0u) << 32) | row[2 * wd];
  const bool hit = (n.attr_simple == 0u && n.ahash_tags != nullptr) ? in_attractor_hashed<kW64>(n, a, y64)
                                                                     : in_attractor<kW64>(n.attr_offset, n.attr_care, n.attr_val, a, y64);
  const bool wrong = !hit && n.r_wrong != 0.0f && in_other_attractor<kW64>(n, a, y64);
  return (hit ? 1u : 0u) | (wrong ? 2u : 0u);
}

// FULL: the tile has all 1024 envs (vector loads/stores); otherwise every access is guarded.
// ASMEM: the attractor table was staged into shared memory (the usual case).
template <bool FULL, bool ASMEM>
__device__ __forceinline__ void tile_step(const StepParams& p, const SlicedSmemLayout& L, uint32_t* scr,
                                          uint32_t* s_surv, float* s_rew, int32_t* s_aoffs, uint32_t* s_aent,
                                          int64_t tile, uint64_t step_ctr, const bool stage, unsigned char* st_state,
                                          unsigned char* st_act, uint64_t* mbar, uint32_t& tma_parity,
                                          const bool pre_drawn, const bool ev_drawn) {
  constexpr bool attr_in_smem = ASMEM;
  const pbn_step_args& a = p.a;
  const NetParams& n = p.n;
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t w = threadIdx.x >> 5;  // warp in tile: owns groups 2w, 2w+1 = rows 8w..8w+7
  const int64_t E = a.n_envs;
  const int64_t e0 = tile * 1024 + 4 * (int64_t)lane;  // local env index of (j = 0, c = 0)
  uint32_t* rows = scr + kScrRows + lane;   // s1 rows (kept for the perturbation phase)
  uint32_t* opl = reinterpret_cast<uint32_t*>(st_state) + lane;  // out planes: the TMA staging buffer is dead after A1
  uint32_t* pl = scr + kScrPl + lane;
  uint32_t* sel0 = scr + kScrSel0 + lane;
  uint32_t* sel1 = scr + kScrSel1 + lane;
  uint32_t* s_stat = scr + kScrStat;

  phase_stamp(a, 0);
  // ---- A0. start the tile's input traffic (consumed after C1, which hides the latency) ---------------
  // full tiles: one thread issues two TMA bulk copies (8 KB*W of state, 1024*BINS action bytes) into the
  // staging buffers; they complete on the CTA's mbarrier, no registers are tied up meanwhile
  if (FULL && threadIdx.x == 0) {
    fence_proxy_async();  // the previous tile's generic-proxy reads of the staging buffers are done
    const uint32_t sbytes = 1024u * 8u * kW64, abytes = 1024u * PBN_BINS;
    mbar_expect_tx(mbar, sbytes + (a.actions != nullptr ? abytes : 0u));
    tma_load_1d(st_state, a.state + tile * 1024 * kW64, sbytes, mbar);
    if (a.actions != nullptr) tma_load_1d(st_act, a.actions + tile * 1024 * PBN_BINS, abytes, mbar);
  }
  uint32_t nfp = 0u;     // 4-bit flip counts of the 8 envs
  uint32_t flips = 0u;
  uint64_t sraw[2][4][kW64];
  uint32_t awraw[2][PBN_BINS];
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    const int64_t e = e0 + 128 * (2 * (int)w + g);
#pragma unroll
    for (int k = 0; k < PBN_BINS; ++k) awraw[g][k] = 0u;
    if (FULL) {
      // state + actions of the tile arrive through the TMA staging buffers (see above)
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
#pragma unroll
        for (int wd = 0; wd < kW64; ++wd) sraw[g][c][wd] = (e + c < E) ? a.state[(e + c) * kW64 + wd] : 0ull;
      }
      if (a.actions != nullptr) {
#pragma unroll
        for (int q = 0; q < 4 * PBN_BINS; ++q) {
          const int64_t env = e + q / PBN_BINS;
          const uint32_t v = (env < E) ? a.actions[e * PBN_BINS + q] : 0u;
          awraw[g][q >> 2] |= v << (8 * (q & 3));
        }
      }
    }
  }

  phase_stamp(a, 1);
  // pre_drawn: done before griddepcontrol.wait.  Otherwise alternate between the CTAs that share an SM (CTAs
  // b, b + #SMs, b + 2 #SMs, ... land on the same SM; the tile parity would not mix: 148 is even)
  unsigned int nsm;
  asm("mov.u32 %0, %%nsmid;" : "=r"(nsm));
  const bool c1_first = !pre_drawn && ((tile / (int64_t)nsm) & 1) == 0;
  if (stage && !c1_first) stage_tables<ASMEM>(n, L, s_surv, s_rew, s_aoffs, s_aent, s_stat);
  phase_stamp(a, 2);
  const uint64_t gid = (uint64_t)(((a.env_offset >> 10) + tile) * 32 + lane);
#if !PBN_INJECTED
  if (!ev_drawn)   // behind the TMA copy
    draw_pert_events(n, scr + kScrEv + threadIdx.x, gid, step_ctr, w, reinterpret_cast<unsigned char*>(scr + kScrPm) + 4u * lane + w);
#endif
  // ---- C1 (even tiles: here, hiding the load latency; odd tiles: after B, so that neighbouring
  //      CTAs of the single wave are in different phases and share the SM's issue slots better)
  if (c1_first) {
    draw_selection_planes<FULL>(a, n, sel0, sel1, gid, step_ctr, e0, w);
    if (stage) stage_tables<ASMEM>(n, L, s_surv, s_rew, s_aoffs, s_aent, s_stat);  // first read after barrier (1)
  }

  phase_stamp(a, 3);
  if (FULL) {
    mbar_wait(mbar, tma_parity);
    tma_parity ^= 1u;
    cta_stamp(a, 1);
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      const int le = 4 * (int)lane + 128 * (2 * (int)w + g);  // env index inside the tile
      const ulonglong2* sp = reinterpret_cast<const ulonglong2*>(st_state + (size_t)le * 8 * kW64);
#pragma unroll
      for (int q = 0; q < 2 * kW64; ++q) {
        const ulonglong2 v = sp[q];
        sraw[g][(2 * q) / kW64][(2 * q) % kW64] = v.x;
        sraw[g][(2 * q + 1) / kW64][(2 * q + 1) % kW64] = v.y;
      }
      if (a.actions != nullptr) {
        const uint32_t* ap = reinterpret_cast<const uint32_t*>(st_act + (size_t)le * PBN_BINS);
#pragma unroll
        for (int k = 0; k < PBN_BINS; ++k) awraw[g][k] = ap[k];
      }
    }
  }
  // ---- A1. apply the interventions, publish the s1 rows -----------------------------------------------
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    const int64_t e = e0 + 128 * (2 * (int)w + g);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      uint32_t fl[kNW];
#pragma unroll
      for (int wd = 0; wd < kNW; ++wd) fl[wd] = 0u;
#pragma unroll
      for (int k = 0; k < PBN_BINS; ++k) {
        const int q = c * PBN_BINS + k;
        const uint32_t act = (awraw[g][q >> 2] >> (8 * (q & 3))) & 0xFFu;
#pragma unroll
        for (int wd = 0; wd < kNW; ++wd) fl[wd] |= shl_clamp(1u, act - 1u - 32u * wd);
      }
      fl[kNW - 1] &= kLastMask;
      uint32_t nf = 0;
#pragma unroll
      for (int wd = 0; wd < kNW; ++wd) nf += __popc(fl[wd]);
      const int i = 4 * g + c;
      nfp |= nf << (4 * i);
      if (FULL || e + c < E) flips += nf;
#pragma unroll
      for (int wd = 0; wd < kNW; ++wd) {
        const uint32_t sw = (uint32_t)(sraw[g][c][wd >> 1] >> (32 * (wd & 1)));
        rows[(wd * 32 + 8 * (int)w + i) * 32] = sw ^ fl[wd];  // row 8w + i of the column
      }
    }
  }
  uint32_t npert = 0u;
#if !PBN_INJECTED
  // Perturbation model A with the kernel's own events (a perturbed env keeps s1 and gets its flips, the update does
  // not apply to it): the flips go into this thread's own s1 rows right here -- the predictors see them only in envs
  // whose function values phase C discards again (pbn_update_part's mux on the event mask) -- so the next state comes
  // out of the ordinary plane pipeline and phase D has nothing to do.
  const bool pert_in_rows = n.pert_rng && n.pert_mode == PBN_PERT_A;   // block-uniform
  if (pert_in_rows) {
    auto flip_row = [&](uint32_t pos) {
      const uint32_t g = pos >> 3, ib = pos & 7u;
      rows[((g >> 5) * 32u + 8u * w + ib) * 32u] ^= 1u << (g & 31u);
      if (FULL || e0 + 128 * (2 * (int)w + (int)(ib >> 2)) + (int)(ib & 3u) < E) ++npert;   // statistics count real envs only
    };
    uint32_t evw[kEvWords];
#pragma unroll
    for (int q = 0; q < kEvWords; ++q) evw[q] = scr[kScrEv + 128 * q + threadIdx.x];
    if (evw[0] != kPreEvOverflow) {
#pragma unroll
      for (int q = 0; q < kEvWords; ++q) {
#pragma unroll 1
        for (uint32_t k = 0; k < kEvPerWord; ++k) {
          const uint32_t pos = (evw[q] >> (kEvBits * k)) & kEvMask;
          if (pos == kEvMask) break;
          flip_row(pos);
        }
      }
    } else {   // more events than the packed list holds (large p): walk the sub-stream again
      const uint32_t s_last = kSurvTable[kSlots];
      uint32_t pert_next = 0u;
      Philox4 pert_blk = {0u, 0u, 0u, 0u};
      int pos = -1;
      while (true) {
        if ((pert_next & 3u) == 0u)
          pert_blk = philox_stream_rk(gid, step_ctr, PBN_RNG_PERTURB, 64u * w + ((pert_next >> 2) & 63u), n.rk);
        const uint32_t u = pick4(pert_blk, pert_next & 3u);
        ++pert_next;
        pos += (u < s_last) ? kSlots + 1 : pert_search(n, u);
        if (pos >= kSlots) break;
        flip_row((uint32_t)pos);
      }
    }
  }
#else
  constexpr bool pert_in_rows = false;
#endif
  phase_stamp(a, 4);
  __syncthreads();  // (1) all 32 s1 rows of the column are in scratch
  phase_stamp(a, 5);

  // ---- B. rows -> bit-planes: this warp produces planes 8w..8w+7 of every word ------------------
#pragma unroll
  for (int wd = 0; wd < kNW; ++wd) {
    uint32_t q8[8];
    transpose_quarter(rows + wd * 32 * 32, w, q8);
#pragma unroll
    for (int i = 0; i < 8; ++i) pl[(wd * 32 + 8 * (int)w + i) * 32] = q8[i];
  }

  phase_stamp(a, 6);
  if (!c1_first && !pre_drawn) draw_selection_planes<FULL>(a, n, sel0, sel1, gid, step_ctr, e0, w);
  __syncthreads();  // (2) all input planes (and selection planes) are in scratch; S1 rows are dead

  // ---- C2. synchronous update of this warp's genes: generated LOP3 trees -> OPL planes ----------
  pbn_update_part(w, pl, opl, sel0, sel1, PBN_SEL2_OF(sel1) pert_in_rows ? scr[kScrPm + lane] : 0u);
  phase_stamp(a, 7);
  __syncthreads();  // (3) all out planes are in scratch
  phase_stamp(a, 8);
  cta_stamp(a, 2);

  // target ids and episode counters of this warp's 8 envs: issued here, consumed in F (E and D hide them)
  uint32_t tg[8];
  uint32_t tt[8];
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    const int64_t e = e0 + 128 * (2 * (int)w + g);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      tg[4 * g + c] = 0xFFFFFFFFu;
      tt[4 * g + c] = 0u;
    }
    if (FULL) {
      if (a.target_id != nullptr) {
        const uint4 v = *reinterpret_cast<const uint4*>(a.target_id + e);
        tg[4 * g] = v.x; tg[4 * g + 1] = v.y; tg[4 * g + 2] = v.z; tg[4 * g + 3] = v.w;
      }
      if (a.t != nullptr) {
        const uint2 v = *reinterpret_cast<const uint2*>(a.t + e);
        tt[4 * g] = v.x & 0xFFFFu; tt[4 * g + 1] = v.x >> 16; tt[4 * g + 2] = v.y & 0xFFFFu; tt[4 * g + 3] = v.y >> 16;
      }
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        if (a.target_id != nullptr && e + c < E) tg[4 * g + c] = (uint32_t)a.target_id[e + c];
        if (a.t != nullptr && e + c < E) tt[4 * g + c] = a.t[e + c];
      }
    }
  }

  // ---- E. bit-planes -> this warp's 8 next-state rows --------------------------------------------
  uint32_t o[8][kNW];
#pragma unroll
  for (int wd = 0; wd < kNW; ++wd) {
    uint32_t q8[8];
    transpose_quarter(opl + wd * 32 * 32, w, q8);
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i][wd] = q8[i];
  }

  phase_stamp(a, 9);
  // ---- D. perturbation (row domain, sparse) ---------------------------------------------------------
  const int pert_mode = n.pert_mode;  // block-uniform
  if (pert_mode != PBN_PERT_NONE && !pert_in_rows) {
#if PBN_INJECTED
    if (a.pert_mask != nullptr) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int64_t env = e0 + 128 * (2 * (int)w + (i >> 2)) + (i & 3);
        uint32_t pm[kNW];
        bool any = false;
#pragma unroll
        for (int wd = 0; wd < kNW; ++wd) {
          pm[wd] = (env < E) ? (uint32_t)(a.pert_mask[env * kW64 + (wd >> 1)] >> (32 * (wd & 1))) : 0u;
          if (wd == kNW - 1) pm[wd] &= kLastMask;
          any = any || pm[wd] != 0u;
          npert += __popc(pm[wd]);
        }
#pragma unroll
        for (int wd = 0; wd < kNW; ++wd) {
          const uint32_t s1w = rows[(wd * 32 + 8 * (int)w + i) * 32];
          if (pert_mode == PBN_PERT_A) o[i][wd] = any ? (s1w ^ pm[wd]) : o[i][wd];
          else if (pert_mode == PBN_PERT_B) o[i][wd] ^= pm[wd];
          else o[i][wd] = bmux(pm[wd], ~s1w, o[i][wd]);
        }
      }
    }
#else
    if (n.pert_rng) {
      // this warp's own event sub-stream: slots gene*8 + row over its 8 rows
      auto apply_event = [&](uint32_t pos) {   // models B and C (model A: see A1)
        const uint32_t g = pos >> 3, ib = pos & 7u;
        const uint32_t m = 1u << (g & 31u), gw = g >> 5;
        if (FULL || e0 + 128 * (2 * (int)w + (int)(ib >> 2)) + (int)(ib & 3u) < E) ++npert;   // statistics count real envs only
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int wd = 0; wd < kNW; ++wd) {
            const bool here = (uint32_t)i == ib;
            const uint32_t mm = (here && (uint32_t)wd == gw) ? m : 0u;
            if (pert_mode == PBN_PERT_B) {
              o[i][wd] ^= mm;
            } else if (here) {
              o[i][wd] = bmux(mm, ~rows[(wd * 32 + 8 * (int)w + i) * 32], o[i][wd]);
            }
          }
      };
      uint32_t evw[kEvWords];
#pragma unroll
      for (int q = 0; q < kEvWords; ++q) evw[q] = scr[kScrEv + 128 * q + threadIdx.x];
      if (evw[0] != kPreEvOverflow) {
        // the usual case: the events were drawn ahead of time (draw_pert_events)
#pragma unroll
        for (int q = 0; q < kEvWords; ++q) {
#pragma unroll 1
          for (uint32_t k = 0; k < kEvPerWord; ++k) {
            const uint32_t pos = (evw[q] >> (kEvBits * k)) & kEvMask;
            if (pos == kEvMask) break;
            apply_event(pos);
          }
        }
      } else {
        const uint32_t s_last = kSurvTable[kSlots];
        uint32_t pert_next = 0u;
        Philox4 pert_blk = {0u, 0u, 0u, 0u};
        int pos = -1;
        while (true) {
          if ((pert_next & 3u) == 0u)
            pert_blk = philox_stream_rk(gid, step_ctr, PBN_RNG_PERTURB, 64u * w + ((pert_next >> 2) & 63u), n.rk);
          const uint32_t u = pick4(pert_blk, pert_next & 3u);
          ++pert_next;
          pos += (u < s_last) ? kSlots + 1 : pert_search(n, u);
          if (pos >= kSlots) break;
          apply_event((uint32_t)pos);
        }
      }
    }
#endif
  }

  phase_stamp(a, 10);
  cta_stamp(a, 4);
  // ---- F. target test, counters, reward, stores ------------------------------------------------------
  uint32_t H = 0u, TR = 0u, VALID = 0u, len_sum = 0u;
  const uint32_t n_attr = (a.target_id != nullptr) ? (uint32_t)n.n_attr : 0u;
  const uint32_t horizon = n.horizon > 0 ? (uint32_t)n.horizon : 0xFFFFFFFFu;
  const bool simple = n.attr_simple != 0u;  // block-uniform
  // ASMEM (compile time): the table sits in shared memory and neither the hash set nor the wrong-attractor term is in
  // play (the host clears the flag otherwise): the out-of-line test below is then not even compiled in
  constexpr bool fast_attr = ASMEM;
  // hash set without wildcard entries and without the wrong-attractor term: probes compacted over the warp (below)
  const bool hash_first = !fast_attr && !simple && n.ahash_tags != nullptr && n.awild_any == 0u && n.r_wrong == 0.0f;
  // ... and single-state targets are tested against their entry in shared memory, no probe at all
  const bool singles = !fast_attr && L.singles_in_smem != 0u;
  uint32_t single = 0u;   // bit i: env i's target is a single-state attractor
  if (singles) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (tg[i] < n_attr && s_aoffs[tg[i]] == 1) single |= 1u << i;
  }
  // Hash-set probes, warp-cooperative: the envs of the warp whose target needs a probe (a fraction of its 256 when most
  // targets are single states) are compacted into a queue -- state words in the warp's own s1 rows, target ids in its
  // own input planes, both dead by now -- and dealt out one per lane: the fingerprint arithmetic and the probe sequence
  // then run once per 32 queued envs at full lane occupancy instead of once per env slot of every thread for the few
  // lanes that need it.  The probing lane writes the verdict over the queued target id.
  uint32_t hq = 0u;       // bit i: env i lies in its target attractor (decided through the queue)
  uint32_t queued = 0u;   // bit i: env i went through the queue
  if (hash_first) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (tg[i] < n_attr && !((single >> i) & 1u)) queued |= 1u << i;
    const uint32_t cnt = (uint32_t)__popc(queued);
    uint32_t incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d);
      if ((int)lane >= d) incl += v;
    }
    const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);   // <= 256: the warp's chunk of rows holds them all
    if (total != 0u) {   // warp-uniform
      uint32_t* qst = scr + kScrRows + 8u * w * 32u;   // word wd of entry q: qst[wd * 1024 + q]
      uint32_t* qtg = scr + kScrPl + 8u * w * 32u;
      uint32_t pos = incl - cnt;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if ((queued >> i) & 1u) {
#pragma unroll
          for (int wd = 0; wd < kNW; ++wd) qst[wd * 1024 + pos] = o[i][wd];
          qtg[pos] = tg[i];
          ++pos;
        }
      __syncwarp();
#pragma unroll 1
      for (uint32_t j = lane; j < total; j += 32u) {
        uint64_t y64[kW64];
#pragma unroll
        for (int wd = 0; wd < kW64; ++wd)
          y64[wd] = ((uint64_t)((2 * wd + 1 < kNW) ? qst[((2 * wd + 1 < kNW) ? 2 * wd + 1 : 0) * 1024 + j] : 0u) << 32) | qst[2 * wd * 1024 + j];
        const int at = (int)qtg[j];
        const uint64_t tag = attr_tag(y64, kW64);
        uint32_t slot = attr_slot(tag, n.ahash_mask);
        uint32_t found = 0u;
#pragma unroll 1
        for (uint32_t probe = 0; probe <= n.ahash_mask; ++probe, slot = (slot + 1u) & n.ahash_mask) {
          const unsigned long long cur = n.ahash_tags[slot];
          if (cur == 0ull) break;
          if (cur == tag && n.ahash_attr[slot] == at) {
            bool same = true;
#pragma unroll
            for (int wd = 0; wd < kW64; ++wd) same = same && n.ahash_state[(size_t)slot * kW64 + wd] == y64[wd];
            if (same) { found = 1u; break; }
          }
        }
        qtg[j] = found;
      }
      __syncwarp();
      pos = incl - cnt;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if ((queued >> i) & 1u) hq |= qtg[pos++] << i;
    }
  }
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    const int64_t e = e0 + 128 * (2 * (int)w + g);
    float rw[4];
    uint32_t hbits = 0u, tbits = 0u, vbits = 0u;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int i = 4 * g + c;
      bool hit = false;
      bool wrong = false;
      if (tg[i] < n_attr) {  // unsigned compare: negative ids never match
        if (!fast_attr) {
          // large attractors (hash set), tables too large for shared memory, or the wrong-attractor reward term.
          // Single-state targets are compared with their entry in shared memory; the hash-set probes of the plain
          // case (no wildcard entries, no wrong-attractor term) were decided through the warp's queue above; anything
          // else goes through the out-of-line test.
          bool decided = false;
          if ((single >> i) & 1u) {
            const uint32_t* ent = s_aent + tg[i] * (2 * kNW);
            uint32_t diff = 0u;
#pragma unroll
            for (int wd = 0; wd < kNW; ++wd) diff |= (o[i][wd] & ent[wd]) ^ ent[kNW + wd];
            hit = diff == 0u;
            decided = true;
          } else if ((queued >> i) & 1u) {
            hit = ((hq >> i) & 1u) != 0u;
            decided = true;
          }
          if (!decided) {
          const uint32_t hw = rare_membership(n, (int)tg[i], o[i][0], o[i][kNW > 1 ? 1 : 0], o[i][kNW > 2 ? 2 : 0], o[i][kNW > 3 ? 3 : 0]);
          hit = (hw & 1u) != 0u;
          wrong = (hw & 2u) != 0u;
          }
        } else if (simple) {
          // one fully specified state per attractor: entry index == attractor id
          const uint32_t* ent = s_aent + tg[i] * (2 * kNW) + kNW;
          uint32_t diff = 0u;
#pragma unroll
          for (int wd = 0; wd < kNW; ++wd) diff |= o[i][wd] ^ ent[wd];
          hit = diff == 0u;
        } else {
          int en = s_aoffs[tg[i]];
          const int en1 = s_aoffs[tg[i] + 1];
#pragma unroll 1
          do {
            const uint32_t* ent = s_aent + en * (2 * kNW);
            uint32_t diff = 0u;
#pragma unroll
            for (int wd = 0; wd < kNW; ++wd) diff |= (o[i][wd] & ent[wd]) ^ ent[kNW + wd];
            hit = hit || diff == 0u;
          } while (++en < en1);
        }
      }
      const uint32_t t1 = min(tt[i] + 1u, 65535u);
      const bool trunc = !hit && t1 >= horizon;
      const uint32_t nf = (nfp >> (4 * i)) & 0xFu;
      rw[c] = s_rew[nf + (hit ? 9u : 0u)];
      if (wrong) rw[c] = __fadd_rn(s_rew[nf], n.r_wrong);
      const bool valid = FULL || (e + c < E);
      hbits |= (hit && valid ? 1u : 0u) << c;
      tbits |= (trunc && valid ? 1u : 0u) << c;
      vbits |= (valid ? 1u : 0u) << c;
      if ((hit || trunc) && valid) len_sum += t1;
      tt[i] = t1;
    }
    H |= hbits << (4 * g);
    TR |= tbits << (4 * g);
    VALID |= vbits << (4 * g);
    const uint32_t hbytes = (hbits * 0x00204081u) & 0x01010101u;
    const uint32_t tbytes = (tbits * 0x00204081u) & 0x01010101u;
    uint64_t y[4][kW64];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int wd = 0; wd < kW64; ++wd)
        y[c][wd] = ((uint64_t)((2 * wd + 1 < kNW) ? o[4 * g + c][(2 * wd + 1 < kNW) ? 2 * wd + 1 : 0] : 0u) << 32) |
                   o[4 * g + c][2 * wd];
    if (FULL) {
      ulonglong2* sp = reinterpret_cast<ulonglong2*>(a.state + e * kW64);
#pragma unroll
      for (int q = 0; q < 2 * kW64; ++q)
        sp[q] = make_ulonglong2(y[(2 * q) / kW64][(2 * q) % kW64], y[(2 * q + 1) / kW64][(2 * q + 1) % kW64]);
      if (a.final_state != nullptr) {
        ulonglong2* fp = reinterpret_cast<ulonglong2*>(a.final_state + e * kW64);
#pragma unroll
        for (int q = 0; q < 2 * kW64; ++q)
          fp[q] = make_ulonglong2(y[(2 * q) / kW64][(2 * q) % kW64], y[(2 * q + 1) / kW64][(2 * q + 1) % kW64]);
      }
      if (a.reward != nullptr) *reinterpret_cast<float4*>(a.reward + e) = make_float4(rw[0], rw[1], rw[2], rw[3]);
      if (a.terminated != nullptr) *reinterpret_cast<uint32_t*>(a.terminated + e) = hbytes;
      if (a.truncated != nullptr) *reinterpret_cast<uint32_t*>(a.truncated + e) = tbytes;
      if (a.t != nullptr)
        *reinterpret_cast<uint2*>(a.t + e) =
            make_uint2(tt[4 * g] | (tt[4 * g + 1] << 16), tt[4 * g + 2] | (tt[4 * g + 3] << 16));
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        if (e + c >= E) continue;
#pragma unroll
        for (int wd = 0; wd < kW64; ++wd) {
          a.state[(e + c) * kW64 + wd] = y[c][wd];
          if (a.final_state != nullptr) a.final_state[(e + c) * kW64 + wd] = y[c][wd];
        }
        if (a.reward != nullptr) a.reward[e + c] = rw[c];
        if (a.terminated != nullptr) a.terminated[e + c] = (uint8_t)((hbits >> c) & 1u);
        if (a.truncated != nullptr) a.truncated[e + c] = (uint8_t)((tbits >> c) & 1u);
        if (a.t != nullptr) a.t[e + c] = (uint16_t)tt[4 * g + c];
      }
    }
  }

  phase_stamp(a, 11);
  // ---- G. auto-reset of finished envs (sparse: scattered writes after the vector stores) ----------
  uint32_t D = (H | TR) & VALID;
  if (a.stats != nullptr) {
    // the per-thread counts are small (8 envs): two 16-bit fields per warp reduction
    const uint32_t x0 = __reduce_add_sync(0xFFFFFFFFu, (uint32_t)__popc(VALID) | ((uint32_t)__popc(H & VALID) << 16));
    const uint32_t x1 = __reduce_add_sync(0xFFFFFFFFu, (uint32_t)__popc(TR & VALID) | (npert << 16));
    const uint32_t x2 = __reduce_add_sync(0xFFFFFFFFu, flips);
    const uint32_t x3 = __reduce_add_sync(0xFFFFFFFFu, len_sum);
    if (lane == 0u) {
      const uint32_t te = x0 >> 16, tr = x1 & 0xFFFFu;
      atomicAdd(&s_stat[PBN_STAT_STEPS], x0 & 0xFFFFu);
      if (te + tr) atomicAdd(&s_stat[PBN_STAT_EPISODES], te + tr);
      if (te) atomicAdd(&s_stat[PBN_STAT_TERMINATED], te);
      if (tr) atomicAdd(&s_stat[PBN_STAT_TRUNCATED], tr);
      if (x3) atomicAdd(&s_stat[PBN_STAT_EP_LEN_SUM], x3);
      if (x2) atomicAdd(&s_stat[PBN_STAT_FLIPS], x2);
      if (x1 >> 16) atomicAdd(&s_stat[PBN_STAT_PERTURBED], x1 >> 16);
    }
  }
  if (a.flags & PBN_STEP_AUTORESET) {
    auto do_reset = [&](int64_t env, const Philox4& r) {
      uint64_t s[kW64];
      int src, tgt;
      if (attr_in_smem) {
        reset_pair(n, r, src, tgt);
        const int o0 = s_aoffs[src];
        const int j = o0 + (int)__umulhi(r.y, (uint32_t)(s_aoffs[src + 1] - o0));
        const uint32_t* ent = s_aent + j * (2 * kNW) + kNW;
#pragma unroll
        for (int wd = 0; wd < kW64; ++wd)
          s[wd] = ((uint64_t)((2 * wd + 1 < kNW) ? ent[(2 * wd + 1 < kNW) ? 2 * wd + 1 : 0] : 0u) << 32) | ent[2 * wd];
      } else {
        reset_draw<kW64>(n, r, s, src, tgt);
      }
#pragma unroll
      for (int wd = 0; wd < kW64; ++wd) a.state[env * kW64 + wd] = s[wd];
      a.target_id[env] = tgt;
      if (a.source_id != nullptr) a.source_id[env] = src;
      a.t[env] = 0;
    };
    // The finished envs of the warp (about 13 of its 256 per step) are dealt out over its lanes, one per lane and
    // trip: a single Philox pass instead of a per-lane serial loop that runs for as long as the unluckiest lane.
    __syncwarp();   // the reset of an env is written by another lane than its outputs in phase F: order the two stores
    const uint32_t cnt = (uint32_t)__popc(D);
    uint32_t incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d);
      if ((int)lane >= d) incl += v;
    }
    const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
    const uint32_t excl = incl - cnt;
    for (uint32_t base = 0; base < total; base += 32u) {   // warp-uniform trip count
      const uint32_t j = base + lane;                      // the job of this lane
      uint32_t L = 0u;                                     // owner: first lane whose inclusive count exceeds j
#pragma unroll
      for (int st = 16; st >= 1; st >>= 1) {
        const uint32_t probe = __shfl_sync(0xFFFFFFFFu, incl, (int)min(L + (uint32_t)st - 1u, 31u));
        if (L + (uint32_t)st - 1u < 32u && probe <= j) L += (uint32_t)st;
      }
      L = min(L, 31u);
      const uint32_t eL = __shfl_sync(0xFFFFFFFFu, excl, (int)L);
      const uint32_t DL = __shfl_sync(0xFFFFFFFFu, D, (int)L);
      if (j < total) {
        uint32_t m = DL;
        for (uint32_t k = j - eL; k != 0u; --k) m &= m - 1u;   // drop the k lowest finished envs of the owner
        const int i = __ffs(m) - 1;
        const int64_t env = tile * 1024 + 4 * (int64_t)L + 128 * (2 * (int)w + (i >> 2)) + (i & 3);
        const Philox4 r = philox_stream_rk((uint64_t)(a.env_offset + env), step_ctr, PBN_RNG_RESET, 0, n.rk);
        do_reset(env, r);
      }
    }
  }
}

#if PBN_BUILD == 0   // the row-format kernels' program (sliced_host.cuh: compile part 0)
// ASMEM: see tile_step.  Two kernels instead of one with a run-time switch: the common one (attractor table in shared
// memory) then contains none of the rare membership code, and its code layout does not move when that code changes
// (measured: 1 us per step of difference from nothing but such a move).
template <bool ASMEM>
__device__ __forceinline__ void step_sliced_body(const StepParams& p, const SlicedSmemLayout& L) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const NetParams& n = p.n;
  const pbn_step_args& a = p.a;
  uint32_t* s_surv = reinterpret_cast<uint32_t*>(smem_raw + L.surv_off);
  float* s_rew = reinterpret_cast<float*>(smem_raw + L.rew_off);
  uint32_t* s_aent = reinterpret_cast<uint32_t*>(smem_raw + L.acare_off);  // [entry][care words | value words]
  int32_t* s_aoffs = reinterpret_cast<int32_t*>(smem_raw + L.aoffs_off);
  uint32_t* scr = reinterpret_cast<uint32_t*>(smem_raw + L.scratch_off);
  unsigned char* st_state = smem_raw + L.stage_state_off;
  unsigned char* st_act = smem_raw + L.stage_act_off;
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_raw + L.mbar_off);
  if (threadIdx.x == 0) mbar_init(mbar, 1u);
  __syncthreads();  // the mbarrier is initialised before anyone polls it
  uint32_t tma_parity = 0u;

  cta_stamp(a, 0);
  const uint64_t step_ctr = effective_step(a);
  const int64_t n_tiles = (a.n_envs + 1023) >> 10;
  bool stage = true;
  bool pre_drawn = false;   // selection planes of the first tile drawn before griddepcontrol.wait
  bool ev_drawn = false;    // ... and its perturbation events
  const int64_t first_tile = (int64_t)blockIdx.x;
  if (a.flags & PBN_STEP_PDL) {
    // Programmatic dependent launch: let the next launch start as SM resources free up, draw this CTA's
    // first tile's selection planes (they depend on nothing the previous launch writes; the device step
    // counter is not bumped by PDL launches), then wait for the previous launch to complete and flush.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // the first tile's inputs were last touched several launches ago (they have left the L2 when the working set
    // exceeds it): pull them in now, the bulk copies after the wait then hit the L2 instead of DRAM
    if ((first_tile + 1) * 1024 <= a.n_envs && threadIdx.x < 4) {
      if (threadIdx.x == 0) l2_prefetch(a.state + first_tile * 1024 * kW64, 1024u * 8u * kW64);
      if (threadIdx.x == 1 && a.actions != nullptr) l2_prefetch(a.actions + first_tile * 1024 * PBN_BINS, 1024u * PBN_BINS);
      if (threadIdx.x == 2 && a.target_id != nullptr) l2_prefetch(a.target_id + first_tile * 1024, 4096u);
      if (threadIdx.x == 3 && a.t != nullptr) l2_prefetch(a.t + first_tile * 1024, 2048u);
    }
    // everything of this CTA's first tile that does not depend on the state: selection planes, perturbation events
    if ((int64_t)blockIdx.x < n_tiles) {
      const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
      const int64_t tile = first_tile;
      const uint64_t gid = (uint64_t)(((a.env_offset >> 10) + tile) * 32 + lane);
      // (measured: letting only every other CTA of an SM draw here and the rest after phase B -- so that their
      // Philox overlaps the others' main phases -- is slower, 23.1 vs 19.1 us: time before the wait is free)
      draw_selection_planes<false>(a, n, scr + kScrSel0 + lane, scr + kScrSel1 + lane, gid, step_ctr,
                                   tile * 1024 + 4 * (int64_t)lane, w);
      pre_drawn = true;
#if !PBN_INJECTED
      draw_pert_events(n, scr + kScrEv + threadIdx.x, gid, step_ctr, w, reinterpret_cast<unsigned char*>(scr + kScrPm) + 4u * lane + w);
      ev_drawn = true;
#endif
    }
    cta_stamp(a, 5);   // (profile builds) pre-wait work done
    asm volatile("griddepcontrol.wait;" ::: "memory");
    cta_stamp(a, 3);   // (profile builds) the previous launch has completed
  }
  for (int64_t tile = first_tile; tile < n_tiles; tile += gridDim.x) {
    const bool full = (tile + 1) * 1024 <= a.n_envs;
    if (full) tile_step<true, ASMEM>(p, L, scr, s_surv, s_rew, s_aoffs, s_aent, tile, step_ctr, stage, st_state, st_act, mbar, tma_parity, pre_drawn, ev_drawn);
    else tile_step<false, ASMEM>(p, L, scr, s_surv, s_rew, s_aoffs, s_aent, tile, step_ctr, stage, st_state, st_act, mbar, tma_parity, pre_drawn, ev_drawn);
    stage = false;
    pre_drawn = false;
    ev_drawn = false;
    phase_stamp(a, 12);
    cta_stamp(a, 6);
    __syncthreads();  // scratch is reused by the next tile; statistics are complete
  }
  if (a.stats != nullptr && threadIdx.x < 7) {
    const uint32_t x = scr[kScrStat + threadIdx.x];
    if (x != 0u) atomicAdd(&a.stats[threadIdx.x], (unsigned long long)x);
  }
  phase_stamp(a, 13);
  cta_stamp(a, 7);
  bump_device_step(a, p.ticket);
  phase_stamp(a, 14);
}

// the host launches pbn_step_sliced when SlicedSmemLayout::attractors_in_smem is set, pbn_step_sliced_gen otherwise
extern "C" __global__ void __launch_bounds__(PBN_THREADS, PBN_MIN_BLOCKS)
pbn_step_sliced(const __grid_constant__ StepParams p, const SlicedSmemLayout L) {
  step_sliced_body<true>(p, L);
}

extern "C" __global__ void __launch_bounds__(PBN_THREADS, PBN_MIN_BLOCKS)
pbn_step_sliced_gen(const __grid_constant__ StepParams p, const SlicedSmemLayout L) {
  step_sliced_body<false>(p, L);
}

#endif  // PBN_BUILD == 0

#if !PBN_INJECTED && (PBN_BUILD == 0 || PBN_BUILD == 2)
// ---- pbn_rollout: S uncontrolled updates (env.step([]) S times, graph_classifier/__init__.py:148; the burn-in of
// the attractor search; compute_ssd_hist's long runs) in ONE launch.  The tile's 1024 states are loaded and
// bit-transposed once, then stay in shared memory as bit-planes: per update only the Philox selection
// planes, the LOP3 trees and the sparse perturbation events remain -- no HBM traffic, no transposes, no
// per-env outputs.  Same random streams as S calls of pbn_step (step counters step_ctr .. step_ctr + S - 1),
// so the final states are bit-identical.
constexpr int kRollPlanes = kNW * 32 * 32;                      // one set of planes [kNW*32][32]
constexpr int kRollSel0 = 2 * kRollPlanes;
constexpr int kRollSel1 = kRollSel0 + PBN_NSEL * 32;
constexpr int kRollEv = kRollSel1 + (PBN_SELBITS - 1) * PBN_NSEL * 32;
constexpr int kRollAny = kRollEv + 128 * kEvWords;              // mode A: rows of the column with an event [32]
constexpr int kRollStat = kRollAny + 32;
constexpr int kRollWords = kRollStat + 8;
constexpr int kRollHist = kRollWords;                           // recording: 2^n_proj histogram bins (u32)
constexpr int kGenesPerWarp = (PBN_N + kWarps - 1) / kWarps;    // recording: genes g = w, w + 4, ... of warp w
// Recording: the shared-memory histogram bins and the per-thread gene counters are u32.  They are flushed into the u64
// accumulators at the end of every tile and, within a tile, after every kRecordFlush recorded updates.  Between two
// flushes a bin gains at most 1024 per recorded update (the tile's envs) and a gene counter at most 32 (its column),
// so they stay below 2^21 * 1024 = 2^31; the warp sum of the 32 gene counters of a gene stays below 2^21 * 1024 too.
constexpr int32_t kRecordFlush = 1 << 21;
// The perturbation count: a thread's u32 count covers at most kPertFold updates of its 8 rows (< 8 * 96 * 2^16 = 3 * 2^24
// events, < 3 * 2^29 for the warp) before it is folded into the block's u64 counter; the count of a call is exact for
// any n_steps and any number of tiles per block.
constexpr int32_t kPertFold = 1 << 16;
static_assert(kRollStat % 2 == 0, "the u64 perturbation counter at kRollStat + 2 must be 8-byte aligned");

template <bool REC> struct RollArgs { using T = RolloutParams; };
template <> struct RollArgs<true> { using T = RecordParams; };
__device__ __forceinline__ const RolloutParams& rollout_of(const RolloutParams& q) { return q; }
__device__ __forceinline__ const RolloutParams& rollout_of(const RecordParams& q) { return q.r; }

// The rollout: REC = false is the plain rollout (pbn_rollout, program 0); REC = true (pbn_rollout_record, program 2) also
// records the states after every update s with s % stride == 0 into the caller's accumulators.  The two are instances of
// one kernel template, looked up by their mangled names (sliced_host.cuh: kRolloutKernel, kRecordKernel): extern "C"
// kernels that inline a shared body compile the plain rollout to different SASS (same instruction count, other
// registers and schedule), a template kernel to the same SASS as before.
template <bool REC>
__global__ void __launch_bounds__(PBN_THREADS, PBN_MIN_BLOCKS) pbn_rollout_sliced(const __grid_constant__ typename RollArgs<REC>::T q) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const RolloutParams& p = rollout_of(q);
  const RecordParams* rec = nullptr;
  if constexpr (REC) rec = &q;
  uint32_t* scr = reinterpret_cast<uint32_t*>(smem_raw);
  const NetParams& n = p.n;
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  const int64_t E = p.n_envs;
  const int64_t n_tiles = (E + 1023) >> 10;
  uint32_t* sel0 = scr + kRollSel0 + lane;
  uint32_t* sel1 = scr + kRollSel1 + lane;
  uint32_t* anym = scr + kRollAny;
  uint32_t* s_stat = scr + kRollStat;   // [0]: the block's real envs; [2..3]: its perturbation count (u64)
  unsigned long long* const s_pert = reinterpret_cast<unsigned long long*>(s_stat + 2);
  const int pert_mode = n.pert_rng ? n.pert_mode : PBN_PERT_NONE;  // block-uniform
  pbn_step_args dummy{};
  if (threadIdx.x < 8) s_stat[threadIdx.x] = 0u;
  // recording (REC): histogram bins [2^n_proj] in shared memory, this thread's column counts of genes w + 4k
  uint32_t* bins = scr + kRollHist;
  uint32_t gcnt[kGenesPerWarp];
  int32_t n_rec = 0;   // recorded updates since the last flush (block-uniform)
  if constexpr (REC) {
    for (int b = threadIdx.x; b < (1 << rec->n_proj); b += kWarps * 32) bins[b] = 0u;   // first added to after a barrier
#pragma unroll
    for (int k = 0; k < kGenesPerWarp; ++k) gcnt[k] = 0u;
  }
  // Record the planes of a completed update (all their writes are ordered before this by a barrier).  vm: the real envs
  // of the column; valid: the real envs among this thread's 8 rows.
  auto record = [&](const uint32_t* planes, uint32_t vm, uint32_t valid) {
    if (rec->gene_on != nullptr) {
#pragma unroll
      for (int k = 0; k < kGenesPerWarp; ++k) {
        const int g = (int)w + kWarps * k;
        if (g < PBN_N) gcnt[k] += __popc(planes[g * 32 + lane] & vm);
      }
    }
    if (rec->hist != nullptr) {
      // bin of row i: bit j = gene proj[j] of the row's env (bit 8w + i of plane proj[j])
      uint32_t idx[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) idx[i] = 0u;
#pragma unroll
      for (int j = 0; j < 12; ++j) {
        if (j < rec->n_proj) {
          const uint32_t x = planes[rec->proj[j] * 32 + lane] >> (8u * w);
#pragma unroll
          for (int i = 0; i < 8; ++i) idx[i] |= ((x >> i) & 1u) << j;
        }
      }
      // a steady state sits on few bins: the lanes of a row that share a bin add once, through their first lane
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const bool ok = (valid >> i) & 1u;
        const uint32_t peers = __match_any_sync(0xFFFFFFFFu, ok ? idx[i] : 0xFFFFFFFFu);
        if (ok && __ffs(peers) - 1 == (int)lane) atomicAdd(&bins[idx[i]], (uint32_t)__popc(peers));
      }
    }
  };
  // add the u32 counters into the u64 accumulators and clear them (every thread, after a barrier)
  auto flush = [&]() {
    if (rec->hist != nullptr) {
      for (int b = threadIdx.x; b < (1 << rec->n_proj); b += kWarps * 32) {
        const uint32_t v = bins[b];
        if (v != 0u) {
          atomicAdd(&rec->hist[b], (unsigned long long)v);
          bins[b] = 0u;
        }
      }
    }
    if (rec->gene_on != nullptr) {
#pragma unroll
      for (int k = 0; k < kGenesPerWarp; ++k) {
        const int g = (int)w + kWarps * k;
        const uint32_t sum = __reduce_add_sync(0xFFFFFFFFu, gcnt[k]);
        if (g < PBN_N && lane == 0u && sum != 0u) atomicAdd(&rec->gene_on[g], (unsigned long long)sum);
        gcnt[k] = 0u;
      }
    }
    n_rec = 0;
  };
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t e0 = tile * 1024 + 4 * (int64_t)lane;
    const uint64_t gid = (uint64_t)(((p.env_offset >> 10) + tile) * 32 + lane);
    uint32_t* cur = scr;                    // current planes
    uint32_t* nxt = scr + kRollPlanes;      // next planes (first: the rows, before the transpose)
    uint32_t valid = 0u;                    // which of this warp's 8 rows are real envs
    uint32_t vm = 0xFFFFFFFFu;              // REC: which of the column's 32 envs are real (bit b: env e0 + 128 (b >> 2) + (b & 3))
    int32_t phase = 0;                      // REC: updates since the last recorded one
    if constexpr (REC) {
      if ((tile + 1) * 1024 > E) {
        vm = 0u;
#pragma unroll
        for (int b = 0; b < 32; ++b) vm |= (e0 + 128 * (b >> 2) + (b & 3) < E ? 1u : 0u) << b;
      }
    }
    // ---- rows of this warp's 8 envs -> scratch
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t env = e0 + 128 * (2 * (int)w + (i >> 2)) + (i & 3);
      const bool ok = env < E;
      valid |= (ok ? 1u : 0u) << i;
#pragma unroll
      for (int wd = 0; wd < kNW; ++wd) {
        const uint64_t v = ok ? p.state[env * kW64 + (wd >> 1)] : 0ull;
        nxt[(wd * 32 + 8 * (int)w + i) * 32 + lane] = (uint32_t)(v >> (32 * (wd & 1)));
      }
    }
    __syncthreads();
    // ---- rows -> bit-planes (this warp: planes 8w..8w+7 of every word)
#pragma unroll
    for (int wd = 0; wd < kNW; ++wd) {
      uint32_t q8[8];
      transpose_quarter(nxt + wd * 32 * 32 + lane, w, q8);
#pragma unroll
      for (int i = 0; i < 8; ++i) cur[(wd * 32 + 8 * (int)w + i) * 32 + lane] = q8[i];
    }
    uint32_t npert = 0u;   // this thread's perturbations since the last fold into s_pert
#pragma unroll 1
    for (int s = 0; s < p.n_steps; ++s) {
      const uint64_t step_ctr = p.step_ctr + (uint64_t)s;
      draw_selection_planes<true>(dummy, n, sel0, sel1, gid, step_ctr, e0, w);
      if (pert_mode != PBN_PERT_NONE) {
        draw_pert_events(n, scr + kRollEv + threadIdx.x, gid, step_ctr, w);
        if (pert_mode == PBN_PERT_A && w == 0u) anym[lane] = 0u;
      }
      __syncthreads();   // planes `cur` complete (transpose / previous update), selection planes drawn
      if constexpr (REC) {
        if (s != 0 && ++phase == rec->stride) {   // `cur` holds the state after update s
          phase = 0;
          record(cur, vm, valid);
          if (++n_rec == kRecordFlush) {
            __syncthreads();
            flush();
            __syncthreads();
          }
        }
      }
      pbn_update_part(w, cur + lane, nxt + lane, sel0, sel1, PBN_SEL2_OF(sel1) 0u);
      if (pert_mode != PBN_PERT_NONE) {
        // this thread's events: (gene, row 8w + ib) of its column
        uint32_t evw[kEvWords];
#pragma unroll
        for (int q = 0; q < kEvWords; ++q) evw[q] = scr[kRollEv + 128 * q + threadIdx.x];
        uint32_t pos_list[kEvCap];
        uint32_t cnt = 0u;
        if (evw[0] != kPreEvOverflow) {
#pragma unroll
          for (int q = 0; q < kEvWords; ++q)
#pragma unroll
            for (uint32_t k = 0; k < kEvPerWord; ++k) {
              const uint32_t pos = (evw[q] >> (kEvBits * k)) & kEvMask;
              pos_list[q * kEvPerWord + k] = pos;
              if (pos != kEvMask && cnt == q * kEvPerWord + k) cnt = q * kEvPerWord + k + 1u;
            }
        }
        const bool overflow = evw[0] == kPreEvOverflow;
        // apply one event to the NEXT planes (after the update of all genes is complete)
        auto flip = [&](uint32_t pos) {
          const uint32_t g = pos >> 3, bit = 8u * w + (pos & 7u);
          uint32_t* word = nxt + g * 32 + lane;
          if (pert_mode == PBN_PERT_C) {
            if ((cur[g * 32 + lane] >> bit) & 1u) atomicAnd(word, ~(1u << bit)); else atomicOr(word, 1u << bit);
          } else {
            atomicXor(word, 1u << bit);
          }
          if ((valid >> (pos & 7u)) & 1u) ++npert;
        };
        if (pert_mode == PBN_PERT_A) {
          // a perturbed step skips the update: rows with an event keep their old bits, then get the flips
          uint32_t M = 0u;
          if (!overflow) {
            for (uint32_t k = 0; k < cnt; ++k) M |= 1u << (8u * w + (pos_list[k] & 7u));
          } else {
            const uint32_t s_last = kSurvTable[kSlots];
            uint32_t pert_next = 0u;
            Philox4 blk = {0u, 0u, 0u, 0u};
            int pos = -1;
            while (true) {
              if ((pert_next & 3u) == 0u) blk = philox_stream_rk(gid, step_ctr, PBN_RNG_PERTURB, 64u * w + ((pert_next >> 2) & 63u), n.rk);
              const uint32_t u = pick4(blk, pert_next & 3u);
              ++pert_next;
              pos += (u < s_last) ? kSlots + 1 : pert_search(n, u);
              if (pos >= kSlots) break;
              M |= 1u << (8u * w + ((uint32_t)pos & 7u));
            }
          }
          if (M) atomicOr(&anym[lane], M);
          __syncthreads();   // all out planes written, all rows-with-events known
          const uint32_t am = anym[lane];
          if (am) {
#pragma unroll 1
            for (int g = (int)w; g < PBN_N; g += kWarps) nxt[g * 32 + lane] = bmux(am, cur[g * 32 + lane], nxt[g * 32 + lane]);
          }
        }
        __syncthreads();     // out planes (and the mode-A restore) complete before the flips
        if (!overflow) {
          for (uint32_t k = 0; k < cnt; ++k) flip(pos_list[k]);
        } else {
          const uint32_t s_last = kSurvTable[kSlots];
          uint32_t pert_next = 0u;
          Philox4 blk = {0u, 0u, 0u, 0u};
          int pos = -1;
          while (true) {
            if ((pert_next & 3u) == 0u) blk = philox_stream_rk(gid, step_ctr, PBN_RNG_PERTURB, 64u * w + ((pert_next >> 2) & 63u), n.rk);
            const uint32_t u = pick4(blk, pert_next & 3u);
            ++pert_next;
            pos += (u < s_last) ? kSlots + 1 : pert_search(n, u);
            if (pos >= kSlots) break;
            flip((uint32_t)pos);
          }
        }
      }
      uint32_t* t = cur; cur = nxt; nxt = t;
      if ((s & (kPertFold - 1)) == kPertFold - 1) {   // fold the count every kPertFold updates (unused without stats)
        const uint32_t np = __reduce_add_sync(0xFFFFFFFFu, npert);
        if (lane == 0u && np) atomicAdd(s_pert, (unsigned long long)np);
        npert = 0u;
      }
    }
    __syncthreads();         // the last update (and its flips) is complete
    if constexpr (REC) {
      if (++phase == rec->stride) record(cur, vm, valid);
    }
    // ---- bit-planes -> this warp's 8 rows -> HBM
    uint32_t o[8][kNW];
#pragma unroll
    for (int wd = 0; wd < kNW; ++wd) {
      uint32_t q8[8];
      transpose_quarter(cur + wd * 32 * 32 + lane, w, q8);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i][wd] = q8[i];
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t env = e0 + 128 * (2 * (int)w + (i >> 2)) + (i & 3);
      if (env < E) {
#pragma unroll
        for (int wd = 0; wd < kW64; ++wd)
          p.state[env * kW64 + wd] = ((uint64_t)((2 * wd + 1 < kNW) ? o[i][(2 * wd + 1 < kNW) ? 2 * wd + 1 : 0] : 0u) << 32) | o[i][2 * wd];
      }
    }
    if (p.stats != nullptr) {
      const uint32_t nv = __reduce_add_sync(0xFFFFFFFFu, (uint32_t)__popc(valid));
      const uint32_t np = __reduce_add_sync(0xFFFFFFFFu, npert);
      if (lane == 0u) {
        atomicAdd(&s_stat[0], nv);
        if (np) atomicAdd(s_pert, (unsigned long long)np);
      }
    }
    __syncthreads();         // scratch is reused by the next tile
    if constexpr (REC) flush();   // (the next tile records after its first barrier)
  }
  if (p.stats != nullptr && threadIdx.x == 0) {
    atomicAdd(&p.stats[PBN_STAT_STEPS], (unsigned long long)s_stat[0] * (unsigned long long)p.n_steps);
    if (*s_pert) atomicAdd(&p.stats[PBN_STAT_PERTURBED], *s_pert);
  }
}

#if PBN_BUILD == 0
template __global__ void pbn_rollout_sliced<false>(const __grid_constant__ RolloutParams q);
#else   // the recording rollout's program (sliced_host.cuh: compile part 2)
template __global__ void pbn_rollout_sliced<true>(const __grid_constant__ RecordParams q);
#endif
#endif

}  // namespace pbn
