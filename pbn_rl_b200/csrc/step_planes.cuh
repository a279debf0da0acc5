// Plane-resident step kernel: the fast path for env state that LIVES on the device as bit-planes.
//
// Resident block (caller-owned DEVICE memory, pbn_resident_words(); written by pbn_resident_import, read back by
// pbn_resident_export): per tile of 1024 consecutive env instances kResRows rows of 32 words, word L of a row =
// column L (the 32 envs  tile*1024 + 128*j + 4*L + c,  bit b = 4*j + c,  j = 0..7, c = 0..3 -- the same env <-> (column,
// bit) map and therefore the same random streams as the row-format kernel, step_sliced.cuh):
//     rows [0, N)            state planes      row g, bit b = gene g of env b
//     rows [N, 2N)           target planes     the state of the env's target attractor (single-state attractors)
//     rows [2N, 2N+8)        target id planes  8-bit id, 255 = no target
//     rows [2N+8, 2N+24)     t planes          16-bit episode step counter
// One 32-bit logic instruction advances 32 envs and nothing is ever transposed: the interventions are scattered into
// the state planes (shared-memory atomics), the predictor functions are generated LOP3 trees, perturbations are
// XOR planes, the target test is N XOR/OR instructions against the target planes, the counters are a bit-sliced
// ripple-carry add and compare; only the per-env results the agent consumes (reward, terminated, truncated) leave
// the plane domain.
//
// Work decomposition: a CTA of WARPS (4 or 8) warps owns one tile.  The genes are split into 8 "parts" (net_update.inc:
// part = selection slot mod 8); a warp draws the selection planes of its part(s) into registers BEFORE
// griddepcontrol.wait (they depend on nothing the previous launch writes) and evaluates the same genes after it, so
// selection planes never leave the register file.  Thread (w, L) handles the per-env inputs/outputs of the column's
// bits [32/WARPS * w, ...).  The tile's block arrives by one TMA bulk copy and leaves by bulk stores.
//   P0  (before the wait) selection planes of the warp's parts; perturbation planes of the step -> O; zero scratch
//       (8-warp variant: warps g / g + 4 share the private blocks of group g, warp g + 4 then walks sub-stream g)
//   P1  TMA load of the tile block -> IN; action bytes -> flips: atomicXor into the state planes (duplicates dropped,
//       so XOR == the OR-mask of the contract); one warp: t' = min(t+1, 65535), t' >= horizon, "has target" plane
//   B1
//   P2  generated LOP3 trees of the warp's genes on s1 -> perturbation -> O; difference to the target planes
//   B2
//   P5  hit / truncated planes -> per-env reward, terminated, truncated (vector stores); statistics; auto-reset:
//       one Philox block per finished env (dealt out over the lanes), then the planes are rewritten gene by gene
//       (warp = genes mod WARPS, lane = column: a gather over the column's finished envs, no atomics)
//   B3  bulk stores of the tile block
// Two instantiations (WARPS = 4 for large batches: 8 CTAs per SM; WARPS = 8 for small ones: half the latency per
// tile) draw identical streams and give identical results.
//
// Random streams: as step_sliced.cuh (SELECT / FIX pool per part, PERTURB sub-streams per 8 slice bits, RESET per env).
// Algorithmic HBM bytes per env-step (SURVEY.md 8d): 33 (N <= 64) / 49.  Bytes this kernel really moves per env-step:
// (2N + 24) / 8 read + written block + BINS action bytes + 6 result bytes (N = 28: 29; N = 70: 50).
#pragma once
#include "pbn_common.cuh"

#ifndef PBN_N
#error "net_gen.cuh and step_sliced.cuh must be included first"
#endif

namespace pbn {

constexpr int kTidPlanes = 8, kTPlanes = 16;
constexpr int kRowTarget = PBN_N, kRowTid = 2 * PBN_N, kRowT = 2 * PBN_N + kTidPlanes;
constexpr int kResRows = 2 * PBN_N + kTidPlanes + kTPlanes;
constexpr int kResTileWords = kResRows * 32;
constexpr uint32_t kNoTarget = 255u;
// shared memory (32-bit words): [dummy row | IN block | O planes | misc | SELX (8-warp variant)]; tables follow at
// PlanesLayout offsets.  The dummy row sits where "gene -1" would be: action value 0 (no-op) needs no test.
constexpr int kPlIn = 32;
constexpr int kPlO = kPlIn + kResTileWords;
constexpr int kPlMisc = kPlO + PBN_N * 32;
constexpr int kPlDiff = kPlMisc, kPlHit = kPlMisc + 32, kPlGe = kPlMisc + 64, kPlHt = kPlMisc + 96, kPlM = kPlMisc + 128;
constexpr int kPlStat = kPlMisc + 160, kPlRew = kPlMisc + 168, kPlMbar = kPlMisc + 192;
constexpr int kPlJobs = kPlMisc + 256;                 // [warp][envs per warp] u16 job list of the auto-reset (2 KB)
constexpr int kPlRinfo = kPlJobs + 512;                // [bit][lane] auto-reset draw of a finished env: source entry | target id << 24 (4 KB)
constexpr int kPlSelx = kPlRinfo + 1024;               // [group][k][lo | hi][lane]: planes of the parts of warps 4..7
constexpr int kPlSelxWords = 4 * PBN_MAXS4 * 2 * 32;
static_assert(2 * (PBN_BINS + 1) <= 24, "reward table does not fit its slot");

__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit_wait_all() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
constexpr int kChainPolls = 1 << 15;   // then the tile falls back to waiting for the whole previous launch

__device__ __forceinline__ void bulk_commit_wait_read() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// One action byte a of an env: if 1 <= a <= N and a differs from the env's earlier bytes p0, p1 (set semantics), toggle
// `bit` in the plane of gene a - 1 (row a of the array at shared byte address xrow0) and add `inc` to cnt; otherwise
// the toggle goes to the dummy row 0.  Branch-free PTX: the compiler builds a branch diamond per action byte, also
// around a predicated atomic.
template <int NPREV>
__device__ __forceinline__ void flip_action(uint32_t xrow0, uint32_t a, uint32_t p0, uint32_t p1, uint32_t bit, uint32_t inc, uint32_t& cnt) {
  if (NPREV == 0) {
    asm volatile("{ .reg .pred p; .reg .u32 t, ad;\n sub.u32 t, %1, 1;\n setp.lt.u32 p, t, %4;\n mad.lo.u32 ad, %1, 128, %2;\n"
                 "@p red.shared.xor.b32 [ad], %3;\n @p add.u32 %0, %0, %5;\n }"
                 : "+r"(cnt) : "r"(a), "r"(xrow0), "r"(bit), "n"(PBN_N), "r"(inc) : "memory");
  } else if (NPREV == 1) {
    asm volatile("{ .reg .pred p; .reg .u32 t, ad;\n sub.u32 t, %1, 1;\n setp.lt.u32 p, t, %4;\n setp.ne.and.u32 p, %1, %6, p;\n"
                 "selp.u32 t, %1, 0, p;\n mad.lo.u32 ad, t, 128, %2;\n red.shared.xor.b32 [ad], %3;\n @p add.u32 %0, %0, %5;\n }"
                 : "+r"(cnt) : "r"(a), "r"(xrow0), "r"(bit), "n"(PBN_N), "r"(inc), "r"(p0) : "memory");
  } else {
    asm volatile("{ .reg .pred p; .reg .u32 t, ad;\n sub.u32 t, %1, 1;\n setp.lt.u32 p, t, %4;\n setp.ne.and.u32 p, %1, %6, p;\n"
                 "setp.ne.and.u32 p, %1, %7, p;\n selp.u32 t, %1, 0, p;\n mad.lo.u32 ad, t, 128, %2;\n red.shared.xor.b32 [ad], %3;\n @p add.u32 %0, %0, %5;\n }"
                 : "+r"(cnt) : "r"(a), "r"(xrow0), "r"(bit), "n"(PBN_N), "r"(inc), "r"(p0), "r"(p1) : "memory");
  }
}

template <int WARPS>
__device__ __forceinline__ void step_planes_body(const StepParams& p, const PlanesLayout& L) {
  constexpr int PARTS = 8 / WARPS;            // evaluation parts per warp (part = w + WARPS * h)
  constexpr int THREADS = 32 * WARPS;
  constexpr int GPT = 8 / WARPS;              // groups of 4 consecutive envs per thread
  constexpr uint32_t kMyBits = (1u << (4 * GPT)) - 1u;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint32_t* const sm = reinterpret_cast<uint32_t*>(smem_raw);
  const pbn_step_args& a = p.a;
  const NetParams& n = p.n;
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  uint32_t* const X = sm + kPlIn + lane;                          // s1 planes   [gene][lane]
  uint32_t* const TG = sm + kPlIn + kRowTarget * 32 + lane;       // target planes
  uint32_t* const TID = sm + kPlIn + kRowTid * 32 + lane;
  uint32_t* const TS = sm + kPlIn + kRowT * 32 + lane;
  uint32_t* const O = sm + kPlO + lane;                   // perturbation planes, then out planes
  uint32_t* const s_stat = sm + kPlStat;
  float* const s_rew = reinterpret_cast<float*>(sm + kPlRew);
  uint64_t* const mbar = reinterpret_cast<uint64_t*>(sm + kPlMbar);
  const uint32_t* const s_aval = reinterpret_cast<const uint32_t*>(smem_raw + L.aval_off);   // [entry][kNW] value words
  const uint32_t* const s_acare = reinterpret_cast<const uint32_t*>(smem_raw + L.acare_off); // [entry][kNW] (generic tables)
  const int32_t* const s_aoffs = reinterpret_cast<const int32_t*>(smem_raw + L.aoffs_off);   // [A+1]
  const uint8_t* const s_eattr = smem_raw + L.eattr_off;                                     // [entry] -> attractor
#if PBN_INJECTED
  const int pm = n.pert_mode;                                   // block-uniform
#else
  const int pm = n.pert_rng ? n.pert_mode : PBN_PERT_NONE;
#endif
  const bool simple = n.attr_simple != 0u;
  const bool has_attr = n.n_attr > 0;
  const int64_t E = a.n_envs;
  const int64_t n_tiles = (E + 1023) >> 10;
  const int64_t first_tile = (int64_t)blockIdx.x;
  // tile-level chaining (PBN_STEP_CHAIN): one epoch word per tile behind the tiles' blocks; a step publishes
  // epoch[tile] = its step counter + 1 once the tile's block is written, the next step of the sequence waits for it
  const bool chain_out = (a.flags & PBN_STEP_CHAIN) != 0u;
  const bool chain_in = chain_out && a.step_ctr != 0u;   // position 0 is launched fully serialised
  uint32_t* const epoch = a.resident + n_tiles * kResTileWords;

  const uint64_t step_ctr = effective_step(a);   // (device counter: the load is issued first, its latency overlaps the staging)
  if (a.flags & PBN_STEP_PDL) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (first_tile < n_tiles && threadIdx.x < 2) {   // warm the L2 with the tile's inputs (coherent, only a hint)
      if (threadIdx.x == 0) l2_prefetch(a.resident + first_tile * kResTileWords, kResTileWords * 4u);
      if (threadIdx.x == 1 && a.actions != nullptr && (first_tile + 1) * 1024 <= E) l2_prefetch(a.actions + first_tile * 1024 * PBN_BINS, 1024u * PBN_BINS);
    }
  }
  // ---- read-only tables of the handle -> shared memory (never written by a step kernel: safe before the wait)
  if (threadIdx.x == 0) mbar_init(mbar, 1u);
  if (threadIdx.x < 2 * (PBN_BINS + 1)) {
    const uint32_t nf = threadIdx.x % (PBN_BINS + 1);
    const bool hit = threadIdx.x >= PBN_BINS + 1;
    const float base = __fadd_rn(n.r_step, __fmul_rn(n.r_action, (float)nf));
    s_rew[threadIdx.x] = __fadd_rn(base, hit ? n.r_success : 0.0f);
  }
  if (threadIdx.x < 8) s_stat[threadIdx.x] = 0u;
  if (L.attr_in_smem) {
    uint32_t* aval = const_cast<uint32_t*>(s_aval);
    uint32_t* acare = const_cast<uint32_t*>(s_acare);
    for (int i = threadIdx.x; i < n.n_attr_states * kNW; i += blockDim.x) {
      const int en = i / kNW, wd = i - en * kNW;
      aval[i] = (uint32_t)(n.attr_val[en * kW64 + (wd >> 1)] >> (32 * (wd & 1)));
      if (!simple) acare[i] = (uint32_t)(n.attr_care[en * kW64 + (wd >> 1)] >> (32 * (wd & 1)));
    }
    for (int i = threadIdx.x; i <= n.n_attr; i += blockDim.x) const_cast<int32_t*>(s_aoffs)[i] = n.attr_offset[i];
    if (!simple)
      for (int at = threadIdx.x; at < n.n_attr; at += blockDim.x)
        for (int en = n.attr_offset[at]; en < n.attr_offset[at + 1]; ++en) const_cast<uint8_t*>(s_eattr)[en] = (uint8_t)at;
  }
  uint32_t parity = 0u;
  bool first = true;

  for (int64_t tile = first_tile; tile < n_tiles; tile += gridDim.x) {
    const int64_t left = E - tile * 1024;                 // envs from the tile's first on
    const bool full = left >= 1024;
    const uint64_t gid = (uint64_t)(((a.env_offset >> 10) + tile) * 32 + lane);
    const int64_t e0 = tile * 1024 + 4 * (int64_t)lane;   // env of (j = 0, c = 0) of this column
    uint32_t VALID = 0xFFFFFFFFu;
    if (!full) {
      VALID = 0u;
      for (int b = 0; b < 32; ++b)
        if (4 * (int)lane + 128 * (b >> 2) + (b & 3) < (int)left) VALID |= 1u << b;
    }
    // ---- P0. everything that does not depend on the previous launch ---------------------------------------
    if (pm != PBN_PERT_NONE) {
      uint4* const o4 = reinterpret_cast<uint4*>(sm + kPlO);
#pragma unroll
      for (int it = 0; it < (PBN_N * 8 + THREADS - 1) / THREADS; ++it) {
        const int i = it * THREADS + (int)threadIdx.x;
        if (i < PBN_N * 8) o4[i] = make_uint4(0u, 0u, 0u, 0u);
      }
    }
    if (threadIdx.x < 32) {
      sm[kPlDiff + lane] = 0u;
      sm[kPlHit + lane] = 0u;
      sm[kPlM + lane] = 0u;
    }
    if (pm != PBN_PERT_NONE) __syncthreads();   // O and M are zero (before the draws: in the 8-warp variant warps 4..7 go straight on to the perturbation walks)
    // selection planes of group w & 3 (slots r = (w & 3) + 4k): the 4-warp variant draws its own; in the 8-warp
    // variant warps g and g + 4 share the private blocks of group g, warp g runs the group's pool and hands the planes
    // of the parts of warps 4..7 over through SELX (read after B1)
    uint32_t lo[PBN_MAXS4], hi[PBN_MAXS4];
#if PBN_INJECTED
#pragma unroll
    for (int k = 0; k < PBN_MAXS4; ++k) {
      const int r = (int)(w & 3u) + 4 * k;
      uint32_t s0 = 0u, s1 = 0u;
      if (r < PBN_NSEL) {
        const uint32_t g = kSelGene[r], K = kSelK[r];
        for (int b = 0; b < 32; ++b) {
          const int64_t env = e0 + 128 * (b >> 2) + (b & 3);
          uint32_t v = (env < E) ? a.sel[env * PBN_N + g] : 0u;
          v = v < K ? v : K - 1u;
          s0 |= (v & 1u) << b;
          s1 |= ((v >> 1) & 1u) << b;
        }
      }
      lo[k] = s0;
      hi[k] = s1;
    }
#else
    if (WARPS == 4) {
      pbn_draw_group(w, gid, step_ctr, n.rk, lo, hi);
    } else if (w >= 4u) {
      // 8-warp variant: warp g + 4 draws the private blocks of group g's odd slots while warp g draws the even ones,
      // hands their results over through SELX (a barrier of the two warps) and goes on to the perturbation walk
      const uint32_t g = w & 3u;
      pbn_draw_group<1>(g, gid, step_ctr, n.rk, lo, hi);
#pragma unroll
      for (int k = 1; k < PBN_MAXS4; k += 2) {
        sm[kPlSelx + ((g * PBN_MAXS4 + k) * 2) * 32 + lane] = lo[k];
        sm[kPlSelx + ((g * PBN_MAXS4 + k) * 2 + 1) * 32 + lane] = hi[k];
      }
      asm volatile("bar.sync %0, 64;" ::"r"(1u + g) : "memory");
    } else {
      pbn_draw_group<0>(w, gid, step_ctr, n.rk, lo, hi);
      asm volatile("bar.sync %0, 64;" ::"r"(1u + w) : "memory");
#pragma unroll
      for (int k = 1; k < PBN_MAXS4; k += 2) {
        lo[k] = sm[kPlSelx + ((w * PBN_MAXS4 + k) * 2) * 32 + lane];
        hi[k] = sm[kPlSelx + ((w * PBN_MAXS4 + k) * 2 + 1) * 32 + lane];
      }
      pbn_draw_group<2>(w, gid, step_ctr, n.rk, lo, hi);   // the group's shared pool, over all its slots
#pragma unroll
      for (int k = 0; k < PBN_MAXS4; ++k) {
        sm[kPlSelx + ((w * PBN_MAXS4 + k) * 2) * 32 + lane] = lo[k];
        sm[kPlSelx + ((w * PBN_MAXS4 + k) * 2 + 1) * 32 + lane] = hi[k];
      }
    }
#endif
    uint32_t npert = 0u;
    if (pm != PBN_PERT_NONE) {
#if PBN_INJECTED
      if (a.pert_mask != nullptr) {
        uint32_t mb = 0u;
        for (int i = 0; i < 4 * GPT; ++i) {
          const uint32_t b = 4u * GPT * w + (uint32_t)i;
          const int64_t env = e0 + 128 * (b >> 2) + (b & 3);
          if (env >= E) continue;
          for (int wd = 0; wd < kNW; ++wd) {
            uint32_t pm = (uint32_t)(a.pert_mask[env * kW64 + (wd >> 1)] >> (32 * (wd & 1)));
            if (wd == kNW - 1) pm &= kLastMask;
            npert += __popc(pm);
            if (pm) mb |= 1u << b;
            while (pm) {
              const int g = 32 * wd + __ffs(pm) - 1;
              pm &= pm - 1u;
              atomicOr(&O[g * 32], 1u << b);
            }
          }
        }
        if (mb) atomicOr(&sm[kPlM + lane], mb);
      }
#else
      // (8-warp variant: warps 4..7 walk the four sub-streams while warps 0..3 are still drawing selection planes)
      if ((WARPS == 8 ? w >= 4u : w < 4u) && n.pert_rng) {
        // sub-stream ws of the column: geometric skipping over the slots gene*8 + (b & 7) of slice bits 8ws..8ws+7
        // (the next event lies pos + 1 + j slots on, j = #{i >= 1 : u < S[i]}: none is left in the rem slots after
        // pos iff u < S[rem] -- one table read settles the usual case, the search runs for real events only)
        const uint32_t ws = w & 3u;
        uint32_t mb = 0u, k = 0u;
        Philox4 blk = philox_stream_rk(gid, step_ctr, PBN_RNG_PERTURB, pert_block(ws, 0u), n.rk);
        int pos = -1;
        uint32_t s_rem = kSurvTable[kSlots];
        while (true) {
          if (k != 0u && (k & 3u) == 0u) blk = philox_stream_rk(gid, step_ctr, PBN_RNG_PERTURB, pert_block(ws, k >> 2), n.rk);
          const uint32_t u = pick4(blk, k & 3u);
          ++k;
          if (u < s_rem) break;
          pos += pert_search(n, u);
          if (pos >= kSlots) break;
          const uint32_t b = 8u * ws + ((uint32_t)pos & 7u);
          atomicOr(&O[(pos >> 3) * 32], 1u << b);
          mb |= 1u << b;
          npert += (VALID >> b) & 1u;
          s_rem = __ldg(n.surv_sliced + (kSlots - 1 - pos));
        }
        if (mb) atomicOr(&sm[kPlM + lane], mb);
      }
#endif
    }
    if (first) {
      __syncthreads();   // mbarrier initialised, tables staged
      if ((a.flags & PBN_STEP_PDL) && !chain_in) asm volatile("griddepcontrol.wait;" ::: "memory");
    }
    // ---- P1. the tile's block; interventions -> state planes; counters ---------------------------------------
    if (threadIdx.x == 0) {
      if (chain_in) {
        const uint32_t want = (uint32_t)step_ctr;
        bool seen = false;
        for (int it = 0; it < kChainPolls && !seen; ++it) {
          seen = ld_acquire_gpu(epoch + tile) == want;
          if (!seen) __nanosleep(64);
        }
        if (!seen) asm volatile("griddepcontrol.wait;" ::: "memory");
      }
      fence_proxy_async();
      mbar_expect_tx(mbar, kResTileWords * 4u);
      tma_load_1d(sm + kPlIn, a.resident + tile * kResTileWords, kResTileWords * 4u, mbar);
    }
    uint32_t act[GPT][PBN_BINS];   // the 4*BINS action bytes of each group of 4 envs
#pragma unroll
    for (int g = 0; g < GPT; ++g) {
#pragma unroll
      for (int k = 0; k < PBN_BINS; ++k) act[g][k] = 0u;
      if (a.actions != nullptr) {
        const int64_t e = e0 + 128 * (GPT * (int)w + g);
        if (full) {
          const uint32_t* ap = reinterpret_cast<const uint32_t*>(a.actions + e * PBN_BINS);
#pragma unroll
          for (int k = 0; k < PBN_BINS; ++k) act[g][k] = __ldg(ap + k);
        } else {
#pragma unroll
          for (int q = 0; q < 4 * PBN_BINS; ++q) {
            const int64_t env = e + q / PBN_BINS;
            const uint32_t v = (env < E) ? a.actions[e * PBN_BINS + q] : 0u;
            act[g][q >> 2] |= v << (8 * (q & 3));
          }
        }
      }
    }
    mbar_wait(mbar, parity);
    parity ^= 1u;
    // flips of this thread's envs: action a >= 1 toggles gene a - 1 (row a of the array that starts at the dummy row);
    // a repeated action of an env is dropped (set semantics), so XOR equals the OR-mask of the contract
    uint32_t nfb[GPT];               // flip counts of each group's 4 envs, one byte per env
    uint32_t flips = 0u;
    {
      const uint32_t xrow0 = smem_u32(sm + kPlIn - 32 + lane);   // row a of this array = plane of gene a - 1
      const uint32_t bit0 = 1u << (4u * GPT * w);
#pragma unroll
      for (int g = 0; g < GPT; ++g) {
        nfb[g] = 0u;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint32_t bit = bit0 << (4 * g + c);
          uint32_t av[PBN_BINS];
#pragma unroll
          for (int k = 0; k < PBN_BINS; ++k) {
            const int q = c * PBN_BINS + k;
            av[k] = __byte_perm(act[g][q >> 2], 0u, 0x4440u + (q & 3));
            if (k == 0) {
              flip_action<0>(xrow0, av[k], 0u, 0u, bit, 1u << (8 * c), nfb[g]);
            } else if (k == 1) {
              flip_action<1>(xrow0, av[k], av[0], 0u, bit, 1u << (8 * c), nfb[g]);
            } else if (k == 2) {
              flip_action<2>(xrow0, av[k], av[0], av[1], bit, 1u << (8 * c), nfb[g]);
            } else {
              bool go = av[k] - 1u < (uint32_t)PBN_N;     // 0 = no-op, values > N are ignored
#pragma unroll
              for (int k2 = 0; k2 < k; ++k2) go = go && av[k2] != av[k];
              if (go) {
                atomicXor(sm + kPlIn - 32 + lane + av[k] * 32u, bit);
                nfb[g] += 1u << (8 * c);
              }
            }
          }
        }
        if (full) {
          flips += nfb[g];
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if ((VALID >> (4 * (GPT * (int)w + g) + c)) & 1u) flips += (nfb[g] >> (8 * c)) & 0xFFu;
        }
      }
      if (full) flips = __dp4a(flips, 0x01010101u, 0u);   // sum of the byte counts
    }
    if (w == WARPS - 1) {
      // t' = min(t + 1, 65535) and GE = (t' >= horizon), bit-sliced; HT = the env has a target
      uint32_t tp[kTPlanes];
      uint32_t sat = 0xFFFFFFFFu;
#pragma unroll
      for (int k = 0; k < kTPlanes; ++k) {
        tp[k] = TS[k * 32];
        sat &= tp[k];
      }
      uint32_t c = ~sat;
#pragma unroll
      for (int k = 0; k < kTPlanes; ++k) {
        const uint32_t nk = tp[k] ^ c;
        c &= tp[k];
        tp[k] = nk;
        TS[k * 32] = nk;
      }
      uint32_t gt = 0u, eq = 0xFFFFFFFFu;
      const uint32_t hz = (uint32_t)n.horizon;
#pragma unroll
      for (int k = kTPlanes - 1; k >= 0; --k) {
        if ((hz >> k) & 1u) eq &= tp[k]; else gt |= eq & tp[k];
      }
      sm[kPlGe + lane] = hz ? (gt | eq) : 0u;
      uint32_t all = 0xFFFFFFFFu;
#pragma unroll
      for (int k = 0; k < kTidPlanes; ++k) all &= TID[k * 32];
      sm[kPlHt + lane] = has_attr ? ~all : 0u;
    }
    __syncthreads();   // B1: s1 planes complete
    // ---- P2. synchronous update of this warp's genes ---------------------------------------------------------
    {
      const uint32_t m = (pm == PBN_PERT_A) ? sm[kPlM + lane] : 0u;
      if (WARPS == 8 && !PBN_INJECTED && w >= 4u) {
#pragma unroll
        for (int k = 0; k < PBN_MAXS4; ++k) {
          lo[k] = sm[kPlSelx + (((w & 3u) * PBN_MAXS4 + k) * 2) * 32 + lane];
          hi[k] = sm[kPlSelx + (((w & 3u) * PBN_MAXS4 + k) * 2 + 1) * 32 + lane];
        }
      }
      uint32_t d = 0u;
#pragma unroll
      for (int h = 0; h < PARTS; ++h) {
        const uint32_t q = w + (uint32_t)WARPS * h;
        if (pm == PBN_PERT_NONE) d |= pbn_eval_part<PBN_PERT_NONE>(q, X, O, TG, m, lo, hi);
        else if (pm == PBN_PERT_A) d |= pbn_eval_part<PBN_PERT_A>(q, X, O, TG, m, lo, hi);
        else if (pm == PBN_PERT_B) d |= pbn_eval_part<PBN_PERT_B>(q, X, O, TG, m, lo, hi);
        else d |= pbn_eval_part<PBN_PERT_C>(q, X, O, TG, m, lo, hi);
      }
      if (d) atomicOr(&sm[kPlDiff + lane], d);
    }
    __syncthreads();   // B2: out planes and target differences complete
    if (!simple && has_attr) {
      // general attractor tables (several states per attractor, wildcards): entry by entry against the out planes
      for (int en = (int)w; en < n.n_attr_states; en += WARPS) {
        const uint32_t aid = s_eattr[en];
        uint32_t m = 0xFFFFFFFFu;
#pragma unroll
        for (int k = 0; k < kTidPlanes; ++k) m &= ((aid >> k) & 1u) ? TID[k * 32] : ~TID[k * 32];
        for (int g = 0; g < PBN_N && m; ++g) {
          const uint32_t care = (s_acare[en * kNW + (g >> 5)] >> (g & 31)) & 1u, val = (s_aval[en * kNW + (g >> 5)] >> (g & 31)) & 1u;
          if (care) m &= val ? O[g * 32] : ~O[g * 32];
        }
        if (m) atomicOr(&sm[kPlHit + lane], m);
      }
      __syncthreads();
    }
    // ---- P5. per-env results ------------------------------------------------------------------------------------
    const uint32_t H = simple ? (~sm[kPlDiff + lane] & sm[kPlHt + lane]) : sm[kPlHit + lane];
    const uint32_t TR = sm[kPlGe + lane] & ~H;
    const uint32_t D = (H | TR) & VALID;
#pragma unroll
    for (int g = 0; g < GPT; ++g) {
      const uint32_t j = GPT * w + g;
      const uint32_t hb = (H >> (4u * j)) & 15u, tb = (TR >> (4u * j)) & 15u;
      const int64_t e = e0 + 128 * (int64_t)j;
      const uint32_t hbytes = (hb * 0x00204081u) & 0x01010101u, tbytes = (tb * 0x00204081u) & 0x01010101u;
      // reward table index of the 4 envs, one byte each: flips + (BINS + 1) * hit
      const uint32_t idx4 = nfb[g] + hbytes * (uint32_t)(PBN_BINS + 1);
      float rw[4];
#pragma unroll
      for (int c = 0; c < 4; ++c)
        rw[c] = *reinterpret_cast<const float*>(reinterpret_cast<const unsigned char*>(s_rew) +
                                                (c == 0 ? (idx4 << 2) & 0x3FCu : (idx4 >> (8 * c - 2)) & 0x3FCu));
      if (full) {
        if (a.reward != nullptr) *reinterpret_cast<float4*>(a.reward + e) = make_float4(rw[0], rw[1], rw[2], rw[3]);
        if (a.terminated != nullptr) *reinterpret_cast<uint32_t*>(a.terminated + e) = hbytes;
        if (a.truncated != nullptr) *reinterpret_cast<uint32_t*>(a.truncated + e) = tbytes;
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (e + c >= E) continue;
          if (a.reward != nullptr) a.reward[e + c] = rw[c];
          if (a.terminated != nullptr) a.terminated[e + c] = (uint8_t)((hb >> c) & 1u);
          if (a.truncated != nullptr) a.truncated[e + c] = (uint8_t)((tb >> c) & 1u);
        }
      }
    }
    const uint32_t mysh = 4u * GPT * w;
    const uint32_t Dm = (D >> mysh) & kMyBits;     // finished envs among this thread's
    uint32_t len_sum = 0u;
    if (w == WARPS - 1 && ((a.flags & PBN_STEP_AUTORESET) || a.stats != nullptr)) {
      // t of the finished envs: summed for the statistics, cleared by the auto-reset
#pragma unroll
      for (int k = 0; k < kTPlanes; ++k) {
        const uint32_t tk = TS[k * 32];
        len_sum += (uint32_t)__popc(tk & D) << k;
        if (a.flags & PBN_STEP_AUTORESET) TS[k * 32] = tk & ~D;
      }
    }
    if (a.stats != nullptr) {
      // per-thread counts are small: two 16-bit fields per warp reduction (terminated | truncated, flips | perturbed)
      const uint32_t mine = kMyBits << mysh;
      const uint32_t x0 = __reduce_add_sync(0xFFFFFFFFu, (uint32_t)__popc(H & VALID & mine) | ((uint32_t)__popc(TR & VALID & mine) << 16));
      const uint32_t x1 = __reduce_add_sync(0xFFFFFFFFu, flips | (npert << 16));
      uint32_t x2 = 0u;
      if (w == WARPS - 1) x2 = __reduce_add_sync(0xFFFFFFFFu, len_sum);
      if (lane == 0u) {
        if (x0 & 0xFFFFu) atomicAdd(&s_stat[PBN_STAT_TERMINATED], x0 & 0xFFFFu);
        if (x0 >> 16) atomicAdd(&s_stat[PBN_STAT_TRUNCATED], x0 >> 16);
        if (x1 & 0xFFFFu) atomicAdd(&s_stat[PBN_STAT_FLIPS], x1 & 0xFFFFu);
        if (x1 >> 16) atomicAdd(&s_stat[PBN_STAT_PERTURBED], x1 >> 16);
        if (x2) atomicAdd(&s_stat[PBN_STAT_EP_LEN_SUM], x2);
      }
    }
    // ---- auto-reset.  R1: the finished envs of the warp are listed in shared memory and dealt out over its lanes (one
    //      Philox pass per 32); the lane leaves its env's draw -- source entry, target id -- at [bit][column].  R2: the
    //      planes are rewritten gene by gene, a warp takes the genes g = w (mod WARPS) of ALL 32 envs of the column:
    //      thread (w, L) gathers the bits of gene g over the finished envs of column L and replaces them in one plain
    //      read-modify-write of its own word -- no atomics (two finished envs of a column share the word, but the
    //      thread owns the whole word), no bank conflicts (lane == bank).  [the first form wrote every bit of a
    //      finished env with a pair of shared-memory atomics: 4 N + 16 per env, a third of the step at N = 70]
    if (a.flags & PBN_STEP_AUTORESET) {
      uint16_t* const jobs = reinterpret_cast<uint16_t*>(sm + kPlJobs) + w * (32 * 4 * GPT);
      uint32_t* const rinfo = sm + kPlRinfo;
      const uint32_t cnt = (uint32_t)__popc(Dm);
      uint32_t incl = cnt;
#pragma unroll
      for (int dd = 1; dd < 32; dd <<= 1) {
        const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, dd);
        if ((int)lane >= dd) incl += v;
      }
      const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
      {
        uint32_t mm = Dm, pos = incl - cnt;
        while (mm) {
          jobs[pos++] = (uint16_t)(lane | ((mysh + (uint32_t)(__ffs(mm) - 1)) << 5));
          mm &= mm - 1u;
        }
      }
      __syncwarp();
      for (uint32_t base = 0; base < total; base += 32u) {   // warp-uniform trip count
        const uint32_t jb = base + lane;                     // the job of this lane
        if (jb < total) {
          const uint32_t code = jobs[jb];
          const uint32_t Lo = code & 31u, b = code >> 5;
          const int64_t env = tile * 1024 + 4 * (int64_t)Lo + 128 * (int64_t)(b >> 2) + (b & 3u);
          const Philox4 r = philox_stream_rk((uint64_t)(a.env_offset + env), step_ctr, PBN_RNG_RESET, 0, n.rk);
          int src, tgt;
          reset_pair(n, r, src, tgt);
          int so, se;
          if (L.attr_in_smem) { so = s_aoffs[src]; se = s_aoffs[src + 1]; }
          else { so = n.attr_offset[src]; se = n.attr_offset[src + 1]; }
          const int js = so + (int)__umulhi(r.y, (uint32_t)(se - so));
          if (a.source_id != nullptr) a.source_id[env] = src;
          rinfo[b * 32u + Lo] = (uint32_t)js | ((uint32_t)tgt << 24);
        }
      }
      __syncthreads();   // every finished env of the tile has its draw
      if (D != 0u) {
        constexpr int GW = (PBN_N + WARPS - 1) / WARPS;      // genes per warp
        constexpr int CH = GW <= 12 ? GW : 8;                // ... gathered CH at a time (registers)
        constexpr int TW = (kTidPlanes + WARPS - 1) / WARPS;  // target id planes per warp
#pragma unroll
        for (int c0 = 0; c0 < GW; c0 += CH) {
          uint32_t ns[CH], nt[CH], ni[TW];
#pragma unroll
          for (int i = 0; i < CH; ++i) { ns[i] = 0u; nt[i] = 0u; }
#pragma unroll
          for (int i = 0; i < TW; ++i) ni[i] = 0u;
          uint32_t mm = D;
#pragma unroll 1
          while (mm) {
            const uint32_t b = (uint32_t)__ffs(mm) - 1u;
            mm &= mm - 1u;
            const uint32_t info = rinfo[b * 32u + lane];
            const uint32_t js = info & 0x00FFFFFFu, tgt = info >> 24;
            const uint32_t to = (uint32_t)(L.attr_in_smem ? s_aoffs[tgt] : n.attr_offset[tgt]);
#pragma unroll
            for (int i = 0; i < CH; ++i) {
              const uint32_t g = w + (uint32_t)(WARPS * (c0 + i));
              if (c0 + i < GW && (GW * WARPS <= PBN_N || g < (uint32_t)PBN_N)) {
                uint32_t sv, tv;
                if (L.attr_in_smem) {
                  sv = s_aval[js * kNW + (g >> 5)];
                  tv = s_aval[to * kNW + (g >> 5)];
                } else {
                  sv = (uint32_t)(n.attr_val[(size_t)js * kW64 + (g >> 6)] >> (32u * ((g >> 5) & 1u)));
                  tv = (uint32_t)(n.attr_val[(size_t)to * kW64 + (g >> 6)] >> (32u * ((g >> 5) & 1u)));
                }
                ns[i] |= ((sv >> (g & 31u)) & 1u) << b;
                nt[i] |= ((tv >> (g & 31u)) & 1u) << b;
              }
            }
            if (c0 == 0) {
#pragma unroll
              for (int i = 0; i < TW; ++i) ni[i] |= ((tgt >> (w + (uint32_t)(WARPS * i))) & 1u) << b;
            }
          }
#pragma unroll
          for (int i = 0; i < CH; ++i) {
            const uint32_t g = w + (uint32_t)(WARPS * (c0 + i));
            if (c0 + i < GW && (GW * WARPS <= PBN_N || g < (uint32_t)PBN_N)) {
              O[g * 32] = (O[g * 32] & ~D) | ns[i];
              TG[g * 32] = (TG[g * 32] & ~D) | nt[i];
            }
          }
          if (c0 == 0) {
#pragma unroll
            for (int i = 0; i < TW; ++i) {
              const uint32_t k = w + (uint32_t)(WARPS * i);
              if (k < (uint32_t)kTidPlanes) TID[k * 32] = (TID[k * 32] & ~D) | ni[i];
            }
          }
        }
      }
    }
    __syncthreads();   // B3: the tile's block is final
    if (a.stats != nullptr && threadIdx.x >= 32u && threadIdx.x < 32u + PBN_N_STATS) {
      // the tile's statistics (every shared-memory counter was updated before B3); warp 1 does it while thread 0 is
      // busy with the block's stores, nobody waits for anybody after B3
      const uint32_t i = threadIdx.x - 32u;
      unsigned long long x = s_stat[i];
      if (i == PBN_STAT_STEPS) x = (unsigned long long)(left < 1024 ? left : 1024);
      if (i == PBN_STAT_EPISODES) x = (unsigned long long)s_stat[PBN_STAT_TERMINATED] + s_stat[PBN_STAT_TRUNCATED];
      __syncwarp(0xFFu);
      s_stat[i] = 0u;
      if (x != 0ull) atomicAdd(&a.stats[i], x);
    }
    if (threadIdx.x == 0) {
      fence_proxy_async();
      uint32_t* gblk = a.resident + tile * kResTileWords;
      bulk_store(gblk, sm + kPlO, PBN_N * 128u);                                   // next states
      if (a.flags & PBN_STEP_AUTORESET)
        bulk_store(gblk + kRowTarget * 32, sm + kPlIn + kRowTarget * 32, (PBN_N + kTidPlanes + kTPlanes) * 128u);
      else
        bulk_store(gblk + kRowT * 32, sm + kPlIn + kRowT * 32, kTPlanes * 128u);   // only the counters changed
      if (chain_out) {
        bulk_commit_wait_all();          // the block is written, not merely read out of shared memory
        fence_proxy_async();
        __threadfence();
        st_release_gpu(epoch + tile, (uint32_t)step_ctr + 1u);
      } else {
        bulk_commit_wait_read();
      }
    }
    first = false;
    if (tile + gridDim.x < n_tiles) __syncthreads();   // the next tile reuses the buffers
  }
  bump_device_step(a, p.ticket);
}

#if PBN_BUILD == 1   // the plane-resident kernels' program (sliced_host.cuh: compile part 1)
extern "C" __global__ void __launch_bounds__(128, PBN_PLANES_MIN_BLOCKS_W4)
pbn_step_planes_w4(const __grid_constant__ StepParams p, const PlanesLayout L) { step_planes_body<4>(p, L); }

extern "C" __global__ void __launch_bounds__(256, PBN_PLANES_MIN_BLOCKS_W8)
pbn_step_planes_w8(const __grid_constant__ StepParams p, const PlanesLayout L) { step_planes_body<8>(p, L); }
#endif  // PBN_BUILD == 1

}  // namespace pbn
