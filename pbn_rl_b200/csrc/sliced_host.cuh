// Host side of the sliced kernel: eligibility, per-network code generation, NVRTC compile
// (with an on-disk cubin cache) and module loading.  Included by pbn_b200.cu only.
#pragma once
#include <dlfcn.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "pbn_common.cuh"

namespace pbn {
namespace jit {

// sources embedded at build time (csrc/Makefile -> embedded_src.inc)
#include "embedded_src.inc"

// Truth table of a predictor over its (ordered) inputs: bit a of the table = value for the input assignment a
// (input j = bit j of a); 2^arity bits in 64-bit words (one word up to 6 inputs).
using Table = std::vector<uint64_t>;

inline bool tab_bit(const Table& t, unsigned a) { return (t[a >> 6] >> (a & 63u)) & 1ull; }
inline void tab_set(Table& t, unsigned a, bool v) {
  if (v) t[a >> 6] |= 1ull << (a & 63u);
}
inline Table tab_make(int k) { return Table((size_t)(k <= 6 ? 1 : (1u << (k - 6))), 0ull); }

struct GenFunc {
  int arity;
  std::vector<int> in;
  Table lut;
  uint32_t cum;   // cumulative selection threshold (2^-32 units) of this predictor within its gene
};

// widest predictor the generated LOP3 trees take (wider ones: thread-per-env kernel)
constexpr int kSlicedMaxArity = 12;

struct GenNet {
  int n_genes = 0, bins = 3, pert_mode = 0;
  bool pert_rng = false;  // perturb_p > 0: the own-RNG specialisation draws perturbation events
  std::vector<std::vector<GenFunc>> funcs;  // per gene
};

// ---- eligibility ---------------------------------------------------------------------------
// The sliced kernels take K in 1..8 predictors per gene: uniform selection among 2, 3 or 4 from 2-bit pairs (exact
// 1-of-3 by rejection), any other probabilities -- and every gene with 5..8 predictors, which makes the network carry
// a third selection plane (PBN_SELBITS == 3) -- by a bit-serial comparison of a 32-bit uniform with the thresholds.
// Predictors of up to kSlicedMaxArity inputs (7 and more: the multi-word tables of pbn_net_desc::wide_lut).
inline bool eligible(const pbn_net_desc* d, std::string* why) {
  if (d->n_genes > 96) {
    if (why) *why = "more than 96 genes";
    return false;
  }
  for (int i = 0; i < d->n_genes; ++i) {
    const int f0 = d->func_offset[i], K = d->func_offset[i + 1] - f0;
    if (K < 1 || K > 8) {
      if (why) *why = "gene with more than 8 predictors";
      return false;
    }
    for (int k = 0; k < K; ++k) {
      if (d->func_arity[f0 + k] > PBN_MAX_ARITY &&
          (d->n_wide <= 0 || !d->wide_inputs || !d->wide_lut_offset || !d->wide_lut || d->func_lut[f0 + k] >= (uint64_t)d->n_wide)) {
        if (why) *why = "wide predictor without its tables";
        return false;
      }
      if (d->func_arity[f0 + k] > kSlicedMaxArity) {
        if (why) *why = "predictor with more than 12 inputs";
        return false;
      }
    }
    for (int k = 0; k + 2 < K; ++k)
      if (d->func_cum[f0 + k] > d->func_cum[f0 + k + 1]) {
        if (why) *why = "selection thresholds of a gene are not non-decreasing";
        return false;
      }
  }
  return true;
}

inline GenNet gen_net_from_desc(const pbn_net_desc* d) {
  GenNet g;
  g.n_genes = d->n_genes;
  g.bins = d->bins;
  g.pert_mode = d->perturb_mode;
  g.pert_rng = d->perturb_p > 0.0;
  g.funcs.resize(d->n_genes);
  for (int i = 0; i < d->n_genes; ++i)
    for (int f = d->func_offset[i]; f < d->func_offset[i + 1]; ++f) {
      GenFunc gf{};
      gf.arity = d->func_arity[f];
      gf.lut = tab_make(gf.arity);
      if (gf.arity > PBN_MAX_ARITY) {  // wide predictor: func_lut holds its index into the wide tables
        const uint64_t v = d->func_lut[f];
        for (int j = 0; j < gf.arity; ++j) gf.in.push_back(d->wide_inputs[v * 16 + j]);
        for (size_t wd = 0; wd < gf.lut.size(); ++wd) gf.lut[wd] = d->wide_lut[d->wide_lut_offset[v] + (int64_t)wd];
      } else {
        for (int j = 0; j < gf.arity; ++j) gf.in.push_back(d->func_inputs[f * PBN_FUNC_INPUT_STRIDE + j]);
        gf.lut[0] = gf.arity >= 6 ? d->func_lut[f] : (d->func_lut[f] & ((1ull << (1u << gf.arity)) - 1ull));
      }
      gf.cum = d->func_cum[f];
      g.funcs[i].push_back(gf);
    }
  return g;
}

// ---- Boolean function -> LOP3 tree -----------------------------------------------------------
struct Expr {
  std::string s;
  int cost;
};

inline std::string plane(int gene) { return "x" + std::to_string(gene); }

// cofactor of t (k variables) with variable j fixed to v: a table over the remaining k - 1 variables
inline Table tab_cofactor(const Table& t, int k, int j, bool v) {
  Table r = tab_make(k - 1);
  unsigned na = 0;
  for (unsigned a = 0; a < (1u << k); ++a) {
    if ((((a >> j) & 1u) != 0u) != v) continue;
    tab_set(r, na, tab_bit(t, a));
    ++na;
  }
  return r;
}

// drop variables the table does not depend on; returns the reduced table, edits vars
inline Table reduce_support(Table lut, std::vector<int>& vars) {
  for (int j = (int)vars.size() - 1; j >= 0; --j) {
    const int k = (int)vars.size();
    Table c0 = tab_cofactor(lut, k, j, false);
    if (c0 != tab_cofactor(lut, k, j, true)) continue;
    lut = c0;
    vars.erase(vars.begin() + j);
  }
  return lut;
}

inline bool tab_complementary(const Table& a, const Table& b, int k) {
  for (unsigned x = 0; x < (1u << k); ++x)
    if (tab_bit(a, x) == tab_bit(b, x)) return false;
  return true;
}

inline Expr synth(Table lut, std::vector<int> vars) {
  lut = reduce_support(lut, vars);
  const int k = (int)vars.size();
  if (k == 0) return {(lut[0] & 1ull) ? "0xFFFFFFFFu" : "0u", 0};
  if (k == 1) return (lut[0] & 3ull) == 2ull ? Expr{plane(vars[0]), 0} : Expr{"(~" + plane(vars[0]) + ")", 1};
  if (k <= 3) {
    unsigned imm = 0;
    for (unsigned t = 0; t < 8; ++t) {
      const unsigned a = (t >> 2) & 1u, b = (t >> 1) & 1u, c = t & 1u;
      const unsigned idx = a | (b << 1) | (k >= 3 ? (c << 2) : 0u);
      imm |= (unsigned)((lut[0] >> idx) & 1ull) << t;
    }
    char buf[160];
    snprintf(buf, sizeof(buf), "lop3<0x%02X>(%s, %s, %s)", imm, plane(vars[0]).c_str(), plane(vars[1]).c_str(),
             plane(vars[k >= 3 ? 2 : 0]).c_str());
    return {buf, 1};
  }
  // Shannon expansion.  Up to 6 variables: on the variable that gives the cheapest pair of cofactors (exhaustive).
  // Beyond: on the variable whose cofactors depend on the fewest variables together (an XOR decomposition first),
  // no search -- the cofactors of real rule tables (sums of products) lose variables quickly.
  std::vector<int> cands;
  if (k <= 6) {
    for (int j = 0; j < k; ++j) cands.push_back(j);
  } else {
    int best_j = 0, best_score = 1 << 30;
    for (int j = 0; j < k; ++j) {
      std::vector<int> r0(vars), r1(vars);
      r0.erase(r0.begin() + j);
      r1.erase(r1.begin() + j);
      const Table c0 = tab_cofactor(lut, k, j, false), c1 = tab_cofactor(lut, k, j, true);
      int score;
      if (tab_complementary(c0, c1, k - 1)) {
        reduce_support(c0, r0);
        score = (int)r0.size() - k;  // one subtree instead of two
      } else {
        reduce_support(c0, r0);
        reduce_support(c1, r1);
        score = (int)r0.size() + (int)r1.size();
      }
      if (score < best_score) best_score = score, best_j = j;
    }
    cands.push_back(best_j);
  }
  Expr best{"", 1 << 30};
  for (int j : cands) {
    const Table lo = tab_cofactor(lut, k, j, false), hi = tab_cofactor(lut, k, j, true);
    std::vector<int> rest(vars);
    rest.erase(rest.begin() + j);
    Expr cand;
    if (tab_complementary(lo, hi, k - 1)) {
      const Expr e0 = synth(lo, rest);
      cand = {"(" + e0.s + " ^ " + plane(vars[j]) + ")", e0.cost + 1};
    } else {
      const Expr e0 = synth(lo, rest), e1 = synth(hi, rest);
      cand = {"bmux(" + plane(vars[j]) + ", " + e1.s + ", " + e0.s + ")", e0.cost + e1.cost + 1};
    }
    if (cand.cost < best.cost) best = cand;
  }
  return best;
}

inline int n_sel_slots(const GenNet& g) {
  int n = 0;
  for (const auto& fs : g.funcs) n += fs.size() > 1 ? 1 : 0;
  return n;
}

// selection planes per slot: 2, or 3 when some gene has more than 4 predictors
inline int sel_bits(const GenNet& g) {
  size_t k = 1;
  for (const auto& fs : g.funcs) k = std::max(k, fs.size());
  return k > 4 ? 3 : 2;
}

inline int scratch_words(const GenNet& g) {
  const int NW = (g.n_genes + 31) / 32;
  // + pre-drawn perturbation events: one packed word per thread (8 N < 255 slots), else two
  // + the model-A event mask of the column (32 words)
  return 2 * NW * 32 * 32 + sel_bits(g) * n_sel_slots(g) * 32 + 8 + 128 * (8 * g.n_genes < 255 ? 1 : 2) + 32;
}

inline int sliced_threads(const GenNet&) { return 128; }  // four warps per 1024-env tile
inline int sliced_min_blocks(const GenNet& g) {
  // one-word states: 7 CTAs per SM (72 registers) -- a 2^20-env step is 1024 tiles on 148 SMs, 6.9 per SM: with 8 slots
  // the CTAs of the next launch pile up on the SMs that finish first (5..8 per SM) and the slowest SM sets the period
  // (measured 16.5 -> 16.1 us per step)
  return g.n_genes <= 32 ? 7 : (g.n_genes <= 64 ? 4 : 2);
}


// Selection groups and evaluation parts: slot r belongs to group r mod 4 and to part r mod 8.  A group draws its
// slots' selection planes (pbn_draw_group: one private Philox block per slot, then the group's shared pool of
// pair-planes for the 1/16 of the 1-of-3 draws that are still rejected -- see step_sliced.cuh "Random streams"); a
// part evaluates its genes (pbn_eval_part, plane-resident kernel).  Single-predictor genes are spread over the
// parts by load.
// A gene's selection is "uniform" when its thresholds are those of 1/K each (what ISPL networks give): the cheap
// pair-plane draw applies.  Anything else is "weighted".
inline bool uniform_selection(const std::vector<GenFunc>& fs) {
  const int K = (int)fs.size();
  if (K > 4) return false;   // 5..8 predictors: always by threshold comparison
  for (int k = 0; k + 1 < K; ++k) {
    const double want = std::floor((double)(k + 1) / K * 4294967296.0 + 0.5);
    if (std::fabs((double)fs[k].cum - want) > 2.0) return false;
  }
  return true;
}

// 1-of-K (K = 5..8) from three selection planes s0, s1, s2 (the unused upper choices repeat the last predictor)
inline std::string mux8(std::vector<std::string> f) {
  while (f.size() < 8) f.push_back(f.back());
  auto mux4 = [&](int b) {
    return "bmux(s1, bmux(s0, " + f[b + 3] + ", " + f[b + 2] + "), bmux(s0, " + f[b + 1] + ", " + f[b] + "))";
  };
  return "bmux(s2, " + mux4(4) + ", " + mux4(0) + ")";
}

inline void generate_parts(const GenNet& g, std::string& u) {
  const int N = g.n_genes;
  char buf[320];
  std::vector<int> part(N, 0), slot_of(N, -1);
  int load[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  int slot = 0;
  for (int i = 0; i < N; ++i)
    if (g.funcs[i].size() > 1) {
      slot_of[i] = slot;
      part[i] = slot & 7;
      load[slot & 7] += (int)g.funcs[i].size() + 2;
      ++slot;
    }
  for (int i = 0; i < N; ++i)
    if (g.funcs[i].size() == 1) {
      int best = 0;
      for (int q = 1; q < 8; ++q)
        if (load[q] < load[best]) best = q;
      part[i] = best;
      load[best] += 1;
    }
  // ---- selection planes of a group: ONE copy of the code for all groups (q is a run-time, warp-uniform value), so
  // that the warps of a tile share their instruction stream; the slot's K is a compile-time constant where the
  // four groups agree on it, else it comes from the kSelK table.
  const int NSEL = slot;
  const int MAXS4 = (NSEL + 3) / 4 > 0 ? (NSEL + 3) / 4 : 1;
  const bool sel3 = sel_bits(g) == 3;
  const int CS = sel3 ? 7 : 3;   // thresholds per slot in kSelCum
  u += "\n#define PBN_CLAIM(k, m3, px, py) { const uint32_t rj_ = lo[k] & hi[k] & (m3); const uint32_t tk_ = rj_ & av; av &= ~rj_; "
       "lo[k] = bmux(tk_, px, lo[k]); hi[k] = bmux(tk_, py, hi[k]); }\n";
  {
    std::string tw, tc;
    int slot_i = 0;
    for (int i = 0; i < N; ++i)
      if (g.funcs[i].size() > 1) {
        tw += (uniform_selection(g.funcs[i]) ? "0, " : "1, ");
        for (int k = 0; k < CS; ++k) {
          snprintf(buf, sizeof(buf), "0x%08Xu, ", k + 1 < (int)g.funcs[i].size() ? g.funcs[i][k].cum : 0xFFFFFFFFu);
          tc += buf;
        }
        ++slot_i;
      }
    if (slot_i == 0) { tw = "0"; tc = "0u"; }
    u += "// slot r draws by threshold comparison (kSelWeighted[r] != 0) against kSelCum[CS r .. CS r + K - 2], CS = 3 (7 with PBN_SELBITS == 3)\n";
    u += "__device__ __constant__ unsigned char kSelWeighted[] = {" + tw + "};\n";
    u += "__device__ __constant__ uint32_t kSelCum[] = {" + tc + "};\n";
  }
  u += "// selection planes of group q (slots r = q + 4k): lo[k] + 2*hi[k] = predictor index, bit-sliced over the column's 32 envs\n";
  u += "// PH: which part of the work (the 8-warp plane-resident kernel splits a group over two warps): -1 everything; 0 / 1 the\n"
       "// private blocks of the even / odd k only; 2 the shared pool only (lo / hi hold the private results of every k)\n";
  u += "#define PBN_DRAWS(k) (PH < 0 || PH == ((k) & 1))\n";
  u += "template <int PH = -1>\n";
  u += "__device__ __forceinline__ void pbn_draw_group(uint32_t q, uint64_t gid, uint64_t step, const uint32_t (&rk)[20],\n"
       "                                               uint32_t (&lo)[PBN_MAXS4], uint32_t (&hi)[PBN_MAXS4]";
  u += sel3 ? ", uint32_t (&h2)[PBN_MAXS4]) {\n" : ") {\n";
  std::vector<int> kof(NSEL, 1), wof(NSEL, 0);
  std::vector<uint32_t> cumof(3 * (NSEL > 0 ? NSEL : 1), 0xFFFFFFFFu);
  for (int i = 0; i < N; ++i)
    if (slot_of[i] >= 0) {
      kof[slot_of[i]] = (int)g.funcs[i].size();
      wof[slot_of[i]] = uniform_selection(g.funcs[i]) ? 0 : 1;
      for (int k = 0; k + 1 < (int)g.funcs[i].size() && k < 3; ++k) cumof[3 * slot_of[i] + k] = g.funcs[i][k].cum;
    }
  std::string any;
  std::vector<std::string> m3(MAXS4);
  for (int k = 0; k < MAXS4; ++k) {
    int Kq[4];
    bool same = true, some3 = false, anyw = false;
    for (int q = 0; q < 4; ++q) {
      const int r = q + 4 * k;
      Kq[q] = r < NSEL ? kof[r] : 1;
      same = same && Kq[q] == Kq[0];
      some3 = some3 || (Kq[q] == 3 && !(r < NSEL && wof[r]));
      anyw = anyw || (r < NSEL && wof[r]);
    }
    snprintf(buf, sizeof(buf), "  if (PBN_DRAWS(%d)) { lo[%d] = 0u; hi[%d] = 0u; }\n", k, k, k);
    u += buf;
    if (sel3) {
      snprintf(buf, sizeof(buf), "  if (PBN_DRAWS(%d)) h2[%d] = 0u;\n", k, k);
      u += buf;
    }
    if (same && Kq[0] == 1) {
      m3[k] = "";
      continue;
    }
    if (same && !anyw) {
      snprintf(buf, sizeof(buf), "  if (PBN_DRAWS(%d)) { const Philox4 A = philox_stream_rk(gid, step, PBN_RNG_SELECT, q + %du, rk);  // K = %d in every group\n", k, 4 * k, Kq[0]);
      u += buf;
      if (Kq[0] == 2) snprintf(buf, sizeof(buf), "    lo[%d] = A.x; }\n", k);
      else if (Kq[0] == 4) snprintf(buf, sizeof(buf), "    lo[%d] = A.x; hi[%d] = A.y; }\n", k, k);
      else snprintf(buf, sizeof(buf), "    const uint32_t rj = A.x & A.y; lo[%d] = bmux(rj, A.z, A.x); hi[%d] = bmux(rj, A.w, A.y); }\n", k, k);
      u += buf;
      m3[k] = Kq[0] == 3 ? "0xFFFFFFFFu" : "";
    } else {
      snprintf(buf, sizeof(buf), "  const uint32_t K%d = (q + %du < %du) ? kSelK[q + %du] : 1u;\n", k, 4 * k, NSEL, 4 * k);
      u += buf;
      if (anyw) {
        snprintf(buf, sizeof(buf), "  const bool W%d = (q + %du < %du) && kSelWeighted[q + %du] != 0;\n", k, 4 * k, NSEL, 4 * k);
        u += buf;
      }
      snprintf(buf, sizeof(buf), "  if (PBN_DRAWS(%d)) {\n", k);
      u += buf;
      if (anyw) {
        if (sel3)
          snprintf(buf, sizeof(buf), "  if (W%d) draw_weighted8(gid, step, rk, q + %du, K%d, kSelCum + 7u * (q + %du), lo[%d], hi[%d], h2[%d]);\n  else ", k, 4 * k, k, 4 * k, k, k, k);
        else
          snprintf(buf, sizeof(buf), "  if (W%d) draw_weighted(gid, step, rk, q + %du, K%d, kSelCum + 3u * (q + %du), lo[%d], hi[%d]);\n  else ", k, 4 * k, k, 4 * k, k, k);
        u += buf;
      } else {
        u += "  ";
      }
      snprintf(buf, sizeof(buf), "if (K%d > 1u) { const Philox4 A = philox_stream_rk(gid, step, PBN_RNG_SELECT, q + %du, rk);\n", k, 4 * k);
      u += buf;
      snprintf(buf, sizeof(buf), "    lo[%d] = A.x; if (K%d == 4u) hi[%d] = A.y;\n", k, k, k);
      u += buf;
      snprintf(buf, sizeof(buf), "    if (K%d == 3u) { const uint32_t rj = A.x & A.y; lo[%d] = bmux(rj, A.z, A.x); hi[%d] = bmux(rj, A.w, A.y); } }\n  }\n", k, k, k);
      u += buf;
      if (some3) {
        if (anyw) snprintf(buf, sizeof(buf), "  const uint32_t m3_%d = (K%d == 3u && !W%d) ? 0xFFFFFFFFu : 0u;\n", k, k, k);
        else snprintf(buf, sizeof(buf), "  const uint32_t m3_%d = K%d == 3u ? 0xFFFFFFFFu : 0u;\n", k, k);
        u += buf;
        snprintf(buf, sizeof(buf), "m3_%d", k);
        m3[k] = buf;
      } else {
        m3[k] = "";
      }
    }
    if (!m3[k].empty()) {
      if (!any.empty()) any += " | ";
      snprintf(buf, sizeof(buf), "(lo[%d] & hi[%d]%s%s)", k, k, m3[k] == "0xFFFFFFFFu" ? "" : " & ", m3[k] == "0xFFFFFFFFu" ? "" : m3[k].c_str());
      any += buf;
    }
  }
  if (!any.empty()) {
    u += "  if (PH < 0 || PH == 2) {\n#pragma unroll 1\n  for (uint32_t i = 0u; i < 1024u; ++i) {  // the group's pool of pair-planes: FIX blocks 1024 q + i\n";
    u += "    if (!__any_sync(0xFFFFFFFFu, (" + any + ") != 0u)) break;\n";
    u += "    const Philox4 P = philox_stream_rk(gid, step, PBN_RNG_FIX, 1024u * q + i, rk);\n    uint32_t av = 0xFFFFFFFFu;\n";
    for (int pass = 0; pass < 2; ++pass) {
      if (pass) u += "    av = 0xFFFFFFFFu;\n";
      for (int k = 0; k < MAXS4; ++k)
        if (!m3[k].empty()) {
          snprintf(buf, sizeof(buf), "    PBN_CLAIM(%d, %s, %s, %s)\n", k, m3[k].c_str(), pass ? "P.z" : "P.x", pass ? "P.w" : "P.y");
          u += buf;
        }
    }
    u += "  }\n  }\n";
  }
  u += "}\n#undef PBN_CLAIM\n#undef PBN_DRAWS\n\n";

  // ---- evaluation of a part's genes in the plane-resident kernel
  u += "// x: s1 planes, o: out planes (on entry: the perturbation planes of the step), tg: target planes; all [gene][lane]\n"
       "// with the lane folded into the pointer.  m: envs of the column with a perturbation event (model A).  Returns the\n"
       "// OR over the part's genes of (next state XOR target state).\n";
  u += "// PM: perturbation model (PBN_PERT_*), a template parameter: the kernel switches once per part\n"
       "#define PBN_FINISH(g, v) { uint32_t v_ = (v); \\\n"
       "    if (PM == 1) v_ = bmux(m, x[(g) * 32], v_) ^ o[(g) * 32]; \\\n"
       "    else if (PM == 2) v_ ^= o[(g) * 32]; \\\n"
       "    else if (PM == 3) v_ = bmux(o[(g) * 32], ~x[(g) * 32], v_); \\\n"
       "    o[(g) * 32] = v_; d |= v_ ^ tg[(g) * 32]; }\n";
  u += "template <int PM>\n";
  u += "// lo / hi: the selection planes of group q mod 4 (pbn_draw_group); slot r of the group sits at index r >> 2\n";
  u += "__device__ __forceinline__ uint32_t pbn_eval_part(uint32_t q, const uint32_t* x, uint32_t* o, const uint32_t* tg, uint32_t m,\n"
       "                                                  const uint32_t (&lo)[PBN_MAXS4], const uint32_t (&hi)[PBN_MAXS4]";
  u += sel3 ? ", const uint32_t (&h2)[PBN_MAXS4]) {\n" : ") {\n";
  u += "  uint32_t d = 0u;\n  (void)m;\n#define X(g) x[(g) * 32]\n";
  for (int q = 0; q < 8; ++q) {
    bool has = false;
    for (int i = 0; i < N; ++i) has = has || part[i] == q;
    if (!has) continue;
    snprintf(buf, sizeof(buf), "  if (q == %du) {\n", q);
    u += buf;
    std::vector<int> used;
    for (int i = 0; i < N; ++i) {
      if (part[i] != q) continue;
      for (const GenFunc& f : g.funcs[i]) {
        std::vector<int> vars(f.in);
        reduce_support(f.lut, vars);
        for (int v : vars)
          if (std::find(used.begin(), used.end(), v) == used.end()) used.push_back(v);
      }
    }
    std::sort(used.begin(), used.end());
    for (int v : used) {
      snprintf(buf, sizeof(buf), "    const uint32_t x%d = X(%d);\n", v, v);
      u += buf;
    }
    for (int i = 0; i < N; ++i) {
      if (part[i] != q) continue;
      const int K = (int)g.funcs[i].size();
      snprintf(buf, sizeof(buf), "    {  // gene %d: %d predictor(s)\n", i, K);
      u += buf;
      std::vector<std::string> names;
      std::vector<std::pair<Table, std::vector<int>>> seen;
      for (int k = 0; k < K; ++k) {
        const GenFunc& f = g.funcs[i][k];
        std::vector<int> vars(f.in);
        const Table red = reduce_support(f.lut, vars);
        int same = -1;
        for (size_t z = 0; z < seen.size(); ++z)
          if (seen[z].first == red && seen[z].second == vars) same = (int)z;
        seen.push_back({red, vars});
        snprintf(buf, sizeof(buf), "f%d", k);
        if (same >= 0) {
          names.push_back(names[same]);
          continue;
        }
        names.push_back(buf);
        const Expr e = synth(f.lut, f.in);
        u += "      const uint32_t " + std::string(buf) + " = " + e.s + ";\n";
      }
      std::string val;
      if (K == 1) {
        val = names[0];
      } else {
        const int k = slot_of[i] >> 2;
        snprintf(buf, sizeof(buf), "      const uint32_t s0 = lo[%d], s1 = hi[%d];\n", k, k);
        u += buf;
        if (K == 2) val = "bmux(s0, " + names[1] + ", " + names[0] + ")", u += "      (void)s1;\n";
        if (K == 3) val = "bmux(s1, " + names[2] + ", bmux(s0, " + names[1] + ", " + names[0] + "))";
        if (K == 4) val = "bmux(s1, bmux(s0, " + names[3] + ", " + names[2] + "), bmux(s0, " + names[1] + ", " + names[0] + "))";
        if (K > 4) {
          snprintf(buf, sizeof(buf), "      const uint32_t s2 = h2[%d];\n", k);
          u += buf;
          val = mux8(names);
        }
      }
      snprintf(buf, sizeof(buf), "      PBN_FINISH(%d, ", i);
      u += buf + val + ")\n    }\n";
    }
    u += "  }\n";
  }
  u += "#undef X\n#undef PBN_FINISH\n  return d;\n}\n";
}

// CTAs per SM the plane-resident kernel is compiled for (register cap = 65536 / (threads * blocks))
inline int planes_min_blocks(const GenNet& g, int warps) {
  if (warps == 4) return g.n_genes <= 32 ? 8 : 4;
  return g.n_genes <= 32 ? 4 : 3;
}

// net_gen.cuh: the constants; net_update.inc: selection tables + pbn_update_part() -- see step_sliced.cuh
inline void generate(const GenNet& g, bool injected, std::string* gen_h, std::string* update_inc) {
  const int N = g.n_genes, NW = (N + 31) / 32, NSEL = n_sel_slots(g);
  char buf[320];
  std::string h;
  h += "// generated by libpbn_b200 for one network: do not edit\n#pragma once\n";
  snprintf(buf, sizeof(buf),
           "#define PBN_N %d\n#define PBN_NW32 %d\n#define PBN_BINS %d\n#define PBN_NSEL %d\n"
           "#define PBN_SCRATCH_WORDS %d\n#define PBN_INJECTED %d\n#define PBN_THREADS %d\n#define PBN_MIN_BLOCKS %d\n",
           N, NW, g.bins, NSEL, scratch_words(g), injected ? 1 : 0, sliced_threads(g), sliced_min_blocks(g));
  h += buf;
  // slots per selection group; plane-resident kernel (step_planes.cuh): CTAs per SM of the two variants
  snprintf(buf, sizeof(buf), "#define PBN_MAXS4 %d\n#define PBN_PLANES_MIN_BLOCKS_W4 %d\n#define PBN_PLANES_MIN_BLOCKS_W8 %d\n",
           (NSEL + 3) / 4 > 0 ? (NSEL + 3) / 4 : 1, planes_min_blocks(g, 4), planes_min_blocks(g, 8));
  h += buf;
  // selection planes per slot (3: some gene has 5..8 predictors)
  snprintf(buf, sizeof(buf), "#define PBN_SELBITS %d\n", sel_bits(g));
  h += buf;
  *gen_h = h;

  // gene -> warp: a gene with a selection slot r is evaluated by the warp that draws slot r (r mod 4);
  // single-predictor genes go to the warp with the fewest functions so far
  std::vector<int> owner(N, 0), slot_of(N, -1);
  int load[4] = {0, 0, 0, 0};
  std::string tg, tk;
  int slot = 0;
  for (int i = 0; i < N; ++i)
    if (g.funcs[i].size() > 1) {
      tg += std::to_string(i) + ", ";
      tk += std::to_string((int)g.funcs[i].size()) + ", ";
      slot_of[i] = slot;
      owner[i] = slot & 3;
      load[slot & 3] += (int)g.funcs[i].size();
      ++slot;
    }
  for (int i = 0; i < N; ++i)
    if (g.funcs[i].size() == 1) {
      int best = 0;
      for (int q = 1; q < 4; ++q)
        if (load[q] < load[best]) best = q;
      owner[i] = best;
      load[best] += 1;
    }
  if (NSEL == 0) {
    tg = "0";
    tk = "1";
  }
  std::string u;
  u += "// generated by libpbn_b200 for one network: do not edit\nnamespace pbn {\n";
  u += "// slot r of the SELECT stream belongs to gene kSelGene[r], which has kSelK[r] predictors\n";
  u += "__device__ __constant__ unsigned char kSelGene[] = {" + tg + "};\n";
  u += "__device__ __constant__ unsigned char kSelK[] = {" + tk + "};\n\n";
  u += "// x: input planes, o: out planes, sel0/sel1: selection planes; all [row][lane], lane folded in\n";
  u += "// keep: envs of the column (bits) that take their input value instead of the update (perturbation model A)\n";
  u += "__device__ __forceinline__ void pbn_update_part(uint32_t w, const uint32_t* x, uint32_t* o,\n"
       "                                                const uint32_t* sel0, const uint32_t* sel1, ";
  u += sel_bits(g) == 3 ? "const uint32_t* sel2, uint32_t keep = 0u) {\n" : "uint32_t keep = 0u) {\n";
  u += "#define X(g) x[(g) * 32]\n";
  for (int q = 0; q < 4; ++q) {
    snprintf(buf, sizeof(buf), "  %sif (w == %du) {\n", q ? "else " : "", q);
    u += buf;
    // load each distinct input plane of this part once
    std::vector<int> used;
    for (int i = 0; i < N; ++i) {
      if (owner[i] != q) continue;
      if (std::find(used.begin(), used.end(), i) == used.end()) used.push_back(i);   // the gene's own plane: keep-mux
      for (const GenFunc& f : g.funcs[i]) {
        std::vector<int> vars(f.in);
        reduce_support(f.lut, vars);
        for (int v : vars)
          if (std::find(used.begin(), used.end(), v) == used.end()) used.push_back(v);
      }
    }
    std::sort(used.begin(), used.end());
    for (int v : used) {
      snprintf(buf, sizeof(buf), "    const uint32_t x%d = X(%d);\n", v, v);
      u += buf;
    }
    for (int i = 0; i < N; ++i) {
      if (owner[i] != q) continue;
      const int K = (int)g.funcs[i].size();
      snprintf(buf, sizeof(buf), "    {  // gene %d: %d predictor(s)\n", i, K);
      u += buf;
      std::vector<std::string> names;
      std::vector<std::pair<Table, std::vector<int>>> seen;
      for (int k = 0; k < K; ++k) {
        const GenFunc& f = g.funcs[i][k];
        std::vector<int> vars(f.in);
        const Table red = reduce_support(f.lut, vars);
        int same = -1;
        for (size_t z = 0; z < seen.size(); ++z)
          if (seen[z].first == red && seen[z].second == vars) same = (int)z;
        seen.push_back({red, vars});
        snprintf(buf, sizeof(buf), "f%d", k);
        if (same >= 0) {
          names.push_back(names[same]);
          continue;
        }
        names.push_back(buf);
        const Expr e = synth(f.lut, f.in);
        u += "      const uint32_t " + std::string(buf) + " = " + e.s + ";\n";
      }
      const std::string dst = "o[" + std::to_string(i * 32) + "] = bmux(keep, " + plane(i) + ", ";
      if (K == 1) {
        u += "      " + dst + names[0] + ");\n    }\n";
        continue;
      }
      snprintf(buf, sizeof(buf), "      const uint32_t s0 = sel0[%d], s1 = sel1[%d];\n", slot_of[i] * 32, slot_of[i] * 32);
      u += buf;
      if (K == 2) u += "      (void)s1;\n      " + dst + "bmux(s0, " + names[1] + ", " + names[0] + "));\n";
      if (K == 3) u += "      " + dst + "bmux(s1, " + names[2] + ", bmux(s0, " + names[1] + ", " + names[0] + ")));\n";
      if (K == 4)
        u += "      " + dst + "bmux(s1, bmux(s0, " + names[3] + ", " + names[2] + "), bmux(s0, " + names[1] + ", " +
             names[0] + ")));\n";
      if (K > 4) {
        snprintf(buf, sizeof(buf), "      const uint32_t s2 = sel2[%d];\n", slot_of[i] * 32);
        u += buf;
        u += "      " + dst + mux8(names) + ");\n";
      }
      u += "    }\n";
    }
    if (q == 0)
      for (int i = N; i < 32 * NW; ++i) {
        snprintf(buf, sizeof(buf), "    o[%d] = 0u;\n", i * 32);
        u += buf;
      }
    u += "  }\n";
  }
  u += "#undef X\n}\n";
  generate_parts(g, u);
  u += "}  // namespace pbn\n";
  *update_inc = u;
}

inline std::string main_source() {
  return "#include \"../../include/pbn_b200.h\"\n#include \"net_gen.cuh\"\n#include \"step_sliced.cuh\"\n#include \"step_planes.cuh\"\n";
}

// ---- NVRTC through dlopen (the library must load on machines without it) ------------------------
struct Nvrtc {
  void* so = nullptr;
  int (*CreateProgram)(void**, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
  int (*CompileProgram)(void*, int, const char* const*) = nullptr;
  int (*GetCUBINSize)(void*, size_t*) = nullptr;
  int (*GetCUBIN)(void*, char*) = nullptr;
  int (*GetProgramLogSize)(void*, size_t*) = nullptr;
  int (*GetProgramLog)(void*, char*) = nullptr;
  int (*DestroyProgram)(void**) = nullptr;
  int (*Version)(int*, int*) = nullptr;
  bool ok() const { return so && CreateProgram && CompileProgram && GetCUBINSize && GetCUBIN && DestroyProgram; }
};

inline Nvrtc& nvrtc() {
  static Nvrtc n;
  if (n.so) return n;
  const char* names[] = {"/usr/local/cuda/lib64/libnvrtc.so.12", "libnvrtc.so.12", "libnvrtc.so", nullptr};
  if (const char* env = getenv("PBN_B200_NVRTC")) n.so = dlopen(env, RTLD_NOW | RTLD_LOCAL);
  for (int i = 0; !n.so && names[i]; ++i) n.so = dlopen(names[i], RTLD_NOW | RTLD_LOCAL);
  if (!n.so) return n;
#define PBN_NVRTC_SYM(field, name) n.field = reinterpret_cast<decltype(n.field)>(dlsym(n.so, name))
  PBN_NVRTC_SYM(CreateProgram, "nvrtcCreateProgram");
  PBN_NVRTC_SYM(CompileProgram, "nvrtcCompileProgram");
  PBN_NVRTC_SYM(GetCUBINSize, "nvrtcGetCUBINSize");
  PBN_NVRTC_SYM(GetCUBIN, "nvrtcGetCUBIN");
  PBN_NVRTC_SYM(GetProgramLogSize, "nvrtcGetProgramLogSize");
  PBN_NVRTC_SYM(GetProgramLog, "nvrtcGetProgramLog");
  PBN_NVRTC_SYM(DestroyProgram, "nvrtcDestroyProgram");
  PBN_NVRTC_SYM(Version, "nvrtcVersion");
#undef PBN_NVRTC_SYM
  return n;
}

inline uint64_t fnv1a(const std::string& s, uint64_t h = 0xcbf29ce484222325ull) {
  for (unsigned char c : s) {
    h ^= c;
    h *= 0x100000001b3ull;
  }
  return h;
}

inline std::string cache_dir() {
  if (const char* env = getenv("PBN_B200_CACHE")) return env;
  Dl_info info;
  std::string dir = ".";
  if (dladdr(reinterpret_cast<void*>(&cache_dir), &info) && info.dli_fname) {
    dir = info.dli_fname;
    const size_t slash = dir.rfind('/');
    dir = slash == std::string::npos ? "." : dir.substr(0, slash);
  }
  return dir + "/_jit_cache";
}

inline bool read_file(const std::string& path, std::vector<char>* out) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) return false;
  fseek(f, 0, SEEK_END);
  const long n = ftell(f);
  fseek(f, 0, SEEK_SET);
  out->resize(n > 0 ? n : 0);
  const bool ok = n > 0 && fread(out->data(), 1, n, f) == (size_t)n;
  fclose(f);
  return ok;
}

inline void write_file_atomic(const std::string& path, const std::vector<char>& data) {
  char tmp[64];
  snprintf(tmp, sizeof(tmp), ".tmp.%d", (int)getpid());
  const std::string t = path + tmp;
  FILE* f = fopen(t.c_str(), "wb");
  if (!f) return;  // cache is best effort
  const bool ok = fwrite(data.data(), 1, data.size(), f) == data.size();
  fclose(f);
  if (ok) rename(t.c_str(), path.c_str());
  else unlink(t.c_str());
}

// PBN_B200_PROFILE=1: compile the %globaltimer phase stamps in (development builds only; flag bit 31 is
// rejected by the ABI otherwise).
inline bool profile_build() {
  const char* env = getenv("PBN_B200_PROFILE");
  return env && env[0] && env[0] != '0';
}

// Mangled names of the two instances of the rollout kernel template (step_sliced.cuh: pbn_rollout_sliced<REC>).
constexpr const char* kRolloutKernel = "_ZN3pbn18pbn_rollout_slicedILb0EEEvNS_8RollArgsIXT_EE1TE";
constexpr const char* kRecordKernel = "_ZN3pbn18pbn_rollout_slicedILb1EEEvNS_8RollArgsIXT_EE1TE";

// Compile (or fetch from the cache) the specialisation; returns 0 or PBN_ERR_JIT with *err set.
// part 0: the row-format kernels (pbn_step_sliced, pbn_rollout_sliced); part 1: the plane-resident
// kernels (pbn_step_planes_w4 / _w8); part 2: the recording rollout (pbn_rollout_sliced<true>, own-RNG only).  Parts 1
// and 2 are compiled and loaded on first use -- separate programs, so that an env that never uses one family never
// pays its compile time.
inline int compile(const GenNet& g, bool injected, int part, std::vector<char>* cubin, std::string* err) {
  std::string gen_h, upd;
  generate(g, injected, &gen_h, &upd);
  const std::string main_src = main_source();
  const bool profile = profile_build();
  const char* opts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo", "-default-device",
                        part == 2 ? "-DPBN_BUILD=2" : part ? "-DPBN_BUILD=1" : "-DPBN_BUILD=0", "-DPBN_PROFILE=1"};
  const int n_opts = profile ? 6 : 5;
  std::string key = gen_h + upd + main_src + kSrc_step_sliced + kSrc_step_planes + kSrc_pbn_common + kSrc_philox + kSrc_pbn_b200_h;
  for (int i = 0; i < n_opts; ++i) key += opts[i];
  char name[64];
  snprintf(name, sizeof(name), "/sliced_%016llx.cubin", (unsigned long long)fnv1a(key));
  const std::string dir = cache_dir(), path = dir + name;
  if (read_file(path, cubin)) return 0;

  Nvrtc& n = nvrtc();
  if (!n.ok()) {
    *err = "libnvrtc.so.12 not found (set PBN_B200_NVRTC) and no cached cubin at " + path;
    return PBN_ERR_JIT;
  }
  const char* hdr_src[] = {kSrc_pbn_b200_h, kSrc_philox, kSrc_pbn_common, kSrc_step_sliced, kSrc_step_planes, gen_h.c_str(), upd.c_str()};
  const char* hdr_name[] = {"../../include/pbn_b200.h", "philox.cuh", "pbn_common.cuh", "step_sliced.cuh", "step_planes.cuh",
                            "net_gen.cuh", "net_update.inc"};
  void* prog = nullptr;
  int rc = n.CreateProgram(&prog, main_src.c_str(), "pbn_sliced.cu", 7, hdr_src, hdr_name);
  if (rc != 0) {
    *err = "nvrtcCreateProgram failed";
    return PBN_ERR_JIT;
  }
  rc = n.CompileProgram(prog, n_opts, opts);
  if (rc != 0) {
    size_t ls = 0;
    std::string log;
    if (n.GetProgramLogSize && n.GetProgramLogSize(prog, &ls) == 0 && ls > 1) {
      log.resize(ls);
      n.GetProgramLog(prog, &log[0]);
    }
    n.DestroyProgram(&prog);
    *err = "nvrtcCompileProgram failed: " + log.substr(0, 1500);
    return PBN_ERR_JIT;
  }
  size_t sz = 0;
  n.GetCUBINSize(prog, &sz);
  cubin->resize(sz);
  n.GetCUBIN(prog, cubin->data());
  n.DestroyProgram(&prog);
  mkdir(dir.c_str(), 0755);
  write_file_atomic(path, *cubin);
  return 0;
}

inline std::vector<uint32_t> sliced_survival(double p, int n_genes) {
  const int slots = 8 * n_genes;  // one sub-stream per (column, warp): 8 rows x N genes
  std::vector<uint32_t> s(slots + 1);
  for (int j = 0; j <= slots; ++j) {
    const double v = std::pow(1.0 - p, (double)j) * 4294967296.0;
    s[j] = v >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)v;
  }
  return s;
}

}  // namespace jit
}  // namespace pbn
