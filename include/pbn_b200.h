/*
 * pbn_b200.h -- C ABI of the B200-native batched Probabilistic Boolean Network environment.
 *
 * This is the drop-in boundary for the hot path of jakub-zarzycki2022/pbn-rl: the PBN
 * environment its agents drive through gym's reset()/step().  In the reference that env is
 * pure Python inside the third-party gym-PBN fork (requirements.txt:11); there is no FFI in
 * the reference, so each entry point below cites the *call site* whose work it takes over.
 * The Python shim pbn_rl_b200/_cabi.py is the only in-tree caller (ctypes); see
 * INTEGRATION.md for the binding a maintainer of the reference would add.
 *
 * Conventions
 *   - Every function returns 0 (PBN_OK) or a negative pbn_status; nothing throws.
 *     pbn_last_error() returns a thread-local message for the last failure.
 *   - All array arguments are DEVICE pointers owned by the caller (e.g. torch tensors'
 *     data_ptr()), except the descriptor/table arguments of pbn_create and
 *     pbn_update_attractors, which are HOST pointers copied during the call.
 *   - Launches go to the caller's stream (a cudaStream_t passed as void*); the library never
 *     synchronises the device.  One handle per GPU; a handle may be used from one thread at
 *     a time.  No global state except the thread-local error string.
 *   - State packing: bit i of a state = gene i (order of the network's Vars: section);
 *     W = 1 64-bit word for N <= 64 genes, W = 2 for N <= 128; env e's words are
 *     state[e*W .. e*W+W-1].
 *
 * One env step (pbn_step), per env instance -- the contract the oracle restates
 * (oracle/pbn_oracle.py: batched_step):
 *   1. flip  = OR over the env's `bins` action bytes a of (1 <= a <= N ? 1<<(a-1) : 0)
 *              (0 = no-op, duplicates do not cancel; bdq_model/__init__.py:82-84,176)
 *      s1    = s XOR flip
 *   2. sel_i = index of the predictor gene i uses this step (injected, or drawn from the
 *              Philox stream with the gene's cumulative selection thresholds)
 *   3. f_i   = LUT[i][sel_i](s1)                        -- synchronous update of all genes
 *   4. perturbation with mask pert (injected, or each gene independently with prob. p):
 *        PBN_PERT_NONE: s' = f
 *        PBN_PERT_A   : s' = pert ? s1 XOR pert : f      (Shmulevich: a perturbed step skips the update)
 *        PBN_PERT_B   : s' = f XOR pert
 *        PBN_PERT_C   : s'_i = pert_i ? NOT s1_i : f_i
 *   5. hit        = target_id in [0, A) and s' matches an entry (care, value) of that attractor
 *   6. t'         = min(t + 1, 65535); terminated = hit;
 *      truncated  = !hit && horizon > 0 && t' >= horizon
 *   7. reward     = (r_step + r_action * popcount(flip)) + (hit ? r_success : wrong ? r_wrong : 0)   [fp32, no FMA]
 *                   wrong = !hit and s' lies in an attractor other than the target (only evaluated when r_wrong != 0;
 *                   upstream gym-PBN's "wrong attractor" penalty, SURVEY.md 8c)
 *   8. with PBN_STEP_AUTORESET, envs with terminated|truncated are re-initialised as by
 *      pbn_reset (new source state / target / t = 0) after their outputs were written.
 *
 * Random streams (own-RNG mode): Philox4x32-10, key = (seed_lo, seed_hi),
 *   counter = (id_lo, id_hi, step_lo, (step_hi & 0xFFFF) | (kind << 28) | (idx << 16)),
 *   kind in {PBN_RNG_SELECT=0, PBN_RNG_PERTURB=1, PBN_RNG_RESET=2, FIX=3 (sliced kernel)}, idx = block index < 4096.
 *   Scalar kernel: id = global env id (env_offset + e).  Gene i uses word i&3 of block
 *   (SELECT, i>>2): sel_i = #{k < K_i-1 : cum[k] <= word}.  Perturbation positions are drawn
 *   by geometric skipping: words of blocks (PERTURB, 0..) in order, skip = #{j in 1..N :
 *   word < survival[j]}, pos += skip + 1, stop when pos >= N.
 *   Sliced kernel: id = global slice-group id; see DESIGN.md section 4 ("Random streams").
 *   Results therefore do not depend on how envs are sharded over GPUs.
 */
#ifndef PBN_B200_H
#define PBN_B200_H

#ifdef __CUDACC_RTC__ /* NVRTC (run-time specialisation of the sliced kernel) has no libc headers */
typedef signed char int8_t;
typedef unsigned char uint8_t;
typedef short int16_t;
typedef unsigned short uint16_t;
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
#else
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define PBN_MAX_GENES 128
#define PBN_MAX_ARITY 6        /* predictors with a 64-bit truth table (func_lut) */
#define PBN_MAX_WIDE_ARITY 16  /* "wide" predictors: multi-word truth tables (wide_lut); up to 12 inputs bit-sliced, beyond: scalar kernel */
#define PBN_MAX_BINS 8
#define PBN_FUNC_INPUT_STRIDE 8

typedef enum {
  PBN_OK = 0,
  PBN_ERR_INVALID = -1,     /* bad argument / descriptor */
  PBN_ERR_CUDA = -2,        /* CUDA runtime error (message has the cudaError string) */
  PBN_ERR_UNSUPPORTED = -3, /* network outside what the requested kernel supports */
  PBN_ERR_NO_ATTRACTORS = -4, /* reset/auto-reset requested before pbn_update_attractors */
  PBN_ERR_JIT = -5          /* run-time specialisation (NVRTC) failed */
} pbn_status;

enum { PBN_PERT_NONE = 0, PBN_PERT_A = 1, PBN_PERT_B = 2, PBN_PERT_C = 3 };
enum { PBN_KERNEL_AUTO = 0, PBN_KERNEL_SCALAR = 1, PBN_KERNEL_SLICED = 2 };
enum { PBN_RNG_SELECT = 0, PBN_RNG_PERTURB = 1, PBN_RNG_RESET = 2 };
enum {
  PBN_STEP_AUTORESET = 1u,
  /* Programmatic dependent launch: the step is launched with programmatic stream serialisation, draws
   * its (state-independent) predictor-selection planes while the previous kernel in the stream is
   * still draining, and only then waits for it (griddepcontrol.wait).  With this flag the launch
   * does NOT increment *step_ctr_dev: pass the position inside the captured sequence as step_ctr
   * and call pbn_advance_counter once at the end of the sequence.  A step enqueued right after its own
   * handle's pbn_advance_counter is launched fully serialised (it reads the counter that launch writes). */
  PBN_STEP_PDL = 2u,
  /* Do not increment *step_ctr_dev when the launch completes (several launches that belong to the same
   * logical step, e.g. the lanes of pbn_step_host, share one counter value). */
  PBN_STEP_NO_COUNT = 4u,
  /* Tile-level chaining of plane-resident steps (args->resident; implies the PBN_STEP_PDL conventions: position in
   * the sequence as step_ctr, pbn_advance_counter at its end).  A launch at position >= 1 does not wait for the
   * whole previous launch: each tile of 1024 envs waits only until the same tile of the previous step of the
   * sequence has published its block (an epoch word per tile in the resident block, release/acquire), so the tails
   * and heads of consecutive steps overlap on the device.  The caller guarantees that (1) the launches of a
   * sequence are consecutive pbn_step calls on one stream for the same block and n_envs, with nothing enqueued
   * between them, and (2) everything else a step reads -- the action buffers of ALL steps of the sequence -- is
   * complete before the sequence's first step is enqueued (open-loop rollouts with pre-sampled actions; not an
   * agent that computes step k+1's actions from step k's results).  Position 0 waits for the whole previous launch.  A tile
   * whose predecessor does not show up within a bounded number of polls falls back to griddepcontrol.wait. */
  PBN_STEP_CHAIN = 8u
};
enum { PBN_UNPACK_U8 = 0, PBN_UNPACK_F32 = 1 };

/* episode statistics accumulated by pbn_step when args->stats != NULL (u64 counters) */
enum {
  PBN_STAT_STEPS = 0,       /* env-steps executed */
  PBN_STAT_EPISODES = 1,    /* episodes finished (terminated | truncated) */
  PBN_STAT_TERMINATED = 2,  /* ... that reached their target attractor */
  PBN_STAT_TRUNCATED = 3,   /* ... that ran into the horizon */
  PBN_STAT_EP_LEN_SUM = 4,  /* sum of t' over finished episodes */
  PBN_STAT_FLIPS = 5,       /* genes flipped by actions */
  PBN_STAT_PERTURBED = 6,   /* genes perturbed */
  PBN_STAT_RESERVED = 7,
  PBN_N_STATS = 8
};

typedef struct pbn_handle pbn_handle;

/* Network + env constants.  Replaces the construction work of
 * gym.make("gym-PBN/BittnerMultiGeneral"|"PBNEnv", ...) (train_BDQ.py:50, train_assa_BQN.py:121-124):
 * the ISPL/logic-function parsing stays in Python, the truth tables arrive here. */
typedef struct {
  int32_t n_genes;              /* N, 1..PBN_MAX_GENES */
  int32_t n_funcs;              /* F = total number of predictor functions */
  const int32_t* func_offset;   /* [N+1] CSR: gene i owns functions func_offset[i]..func_offset[i+1]-1 */
  const uint8_t* func_arity;    /* [F] 0..PBN_MAX_ARITY */
  const uint8_t* func_inputs;   /* [F*8] gene index feeding bit j of the truth-table index */
  const uint64_t* func_lut;     /* [F] truth table: bit a = value for input assignment a */
  const uint32_t* func_cum;     /* [F] cumulative selection thresholds in 2^-32 units (last of a gene ignored) */
  const uint32_t* survival;     /* [N+1] floor((1-p)^j 2^32) or NULL: computed from perturb_p */
  int32_t bins;                 /* action bytes per env per step, 1..PBN_MAX_BINS (bdq_model/utils.py:48: 3) */
  int32_t horizon;              /* steps until truncation; 0 = never (train_BDQ.py:50: 20) */
  int32_t perturb_mode;         /* PBN_PERT_* */
  double perturb_p;             /* per-gene perturbation probability */
  float r_success, r_step, r_action;
  uint64_t seed;                /* Philox key */
  int32_t device;               /* CUDA device ordinal */
  int32_t kernel;               /* PBN_KERNEL_* */
  /* Wide predictors (arity 7..PBN_MAX_WIDE_ARITY), e.g. the inline logic_functions of model_tester.py:97-341
   * and train_control_gbdq.py:45-72.  Function f is wide iff func_arity[f] > PBN_MAX_ARITY; then
   * func_lut[f] holds its index v into these tables and func_inputs[f*8..] is ignored.  n_wide = 0 and
   * NULL pointers when the network has none. */
  int32_t n_wide;
  int32_t reserved0;
  const uint8_t* wide_inputs;       /* [n_wide*16] gene index feeding bit j of the truth-table index */
  const int32_t* wide_lut_offset;   /* [n_wide+1] offsets into wide_lut, in 64-bit words */
  const uint64_t* wide_lut;         /* truth tables: bit a of table v = wide_lut[off[v] + a/64] >> (a%64) */
  float r_wrong;                    /* reward term for ending a step in an attractor that is not the target; 0 = none */
  float reserved1;
} pbn_net_desc;

/* Arguments of one step over n_envs instances (device pointers). */
typedef struct {
  uint64_t* state;              /* [E*W] in/out */
  const uint8_t* actions;       /* [E*bins] in; NULL = no interventions (env.step([]), graph_classifier/__init__.py:148) */
  int32_t* target_id;           /* [E] in (written on auto-reset); NULL = no target test */
  int32_t* source_id;           /* [E] or NULL; written on auto-reset */
  uint16_t* t;                  /* [E] in/out episode step counters (env.n_steps) */
  float* reward;                /* [E] out */
  uint8_t* terminated;          /* [E] out */
  uint8_t* truncated;           /* [E] out */
  uint64_t* final_state;        /* [E*W] or NULL; with auto-reset: the pre-reset next state of every env */
  const uint64_t* pert_mask;    /* [E*W] injected perturbation masks (pbn_step_injected), may be NULL = none */
  const uint8_t* sel;           /* [E*N] injected predictor choices (pbn_step_injected) */
  unsigned long long* stats;    /* [PBN_N_STATS] or NULL */
  uint64_t* step_ctr_dev;       /* device counter or NULL.  If given, the step uses step_ctr + *step_ctr_dev
                                   and the launch increments *step_ctr_dev when it completes, so a CUDA graph
                                   of captured steps keeps advancing the random streams on every replay */
  uint64_t step_ctr;            /* Philox step counter; the caller increments it every step */
  int64_t env_offset;           /* global id of env 0 of this call (multiple of 1024) */
  int64_t n_envs;               /* E */
  uint32_t flags;               /* PBN_STEP_* */
  uint32_t reserved;
  uint32_t* resident;           /* [pbn_resident_words()] plane-resident env state (see pbn_resident_import) or NULL.
                                   When given, it replaces state / target_id / t (which must be NULL): the step
                                   reads and writes the env state in the resident block; the per-env results
                                   reward / terminated / truncated are produced as usual */
} pbn_step_args;

/* gym.make(...) construction: upload truth tables and constants, pick the kernel. */
int pbn_create(const pbn_net_desc* desc, pbn_handle** out);
void pbn_destroy(pbn_handle* h);

/* (Re-)upload the attractor table: env.all_attractors may grow during training
 * (bdq_model/__init__.py:182-184); env.setTarget / in_target / is_attracting_state
 * (model_tester.py:614-616, graph_classifier/__init__.py:129) read it.
 * attr_offset[A+1] CSR into care/value [S*W] (HOST pointers).  pair_cum: [A*A] cumulative
 * u32 thresholds over (source*A + target) pairs for reset sampling -- the curriculum of
 * env.rework_probas (bdq_model/__init__.py:203) -- or NULL = uniform over source != target.
 * The device tables are allocated with spare capacity and updated IN PLACE by copies on `stream` (ordered
 * after the steps already enqueued there): their addresses stay valid, so launches and CUDA graphs captured
 * earlier never see freed memory.  Only when a table outgrows its capacity does the call synchronise `stream`
 * and reallocate (graphs captured before that must be re-captured); table sizes travel in the kernel
 * parameters, so a captured graph keeps using the sizes it was captured with.  Not legal during stream capture. */
int pbn_update_attractors(pbn_handle* h, const int32_t* attr_offset, const uint64_t* care,
                          const uint64_t* value, int32_t n_attractors, const uint32_t* pair_cum,
                          void* stream);

/* env.step(action) for every instance (bdq_model/__init__.py:177; ddqn_per/__init__.py:354),
 * randomness from the handle's Philox stream.  args->sel and args->pert_mask must be NULL. */
int pbn_step(pbn_handle* h, const pbn_step_args* args, void* stream);

/* Host buffers of pbn_step_host: what a caller of the reference's CPU env holds per step -- the
 * action it passes to env.step (bdq_model/__init__.py:176-177) and the tuple it gets back
 * (state, reward, terminated, truncated).  HOST pointers (page-locked memory for the copies to
 * overlap; pageable memory works but serialises); any output may be NULL = not wanted. */
typedef struct {
  const uint8_t* actions;   /* HOST [E*bins] in; NULL = no interventions */
  uint8_t* actions_dev;     /* DEVICE [E*bins] staging buffer, caller-owned (required with actions) */
  uint64_t* state;          /* HOST [E*W] out: args->state after the step (after auto-reset, if enabled) */
  float* reward;            /* HOST [E] out */
  uint8_t* terminated;      /* HOST [E] out */
  uint8_t* truncated;       /* HOST [E] out */
  int32_t n_chunks;         /* number of lanes; 0 = library default */
  int32_t reserved;
  /* Compact forms of the same results (fewer PCIe bytes per env-step); page-locked memory only. */
  uint32_t* state32;        /* HOST [E] out: the state word narrowed to 32 bits; networks with N <= 32 only */
  uint8_t* done;            /* HOST [E] out: terminated | truncated << 1 */
  /* The smallest form, 6 bytes per env-step over PCIe (N <= 30, bins == 3; page-locked memory): */
  uint32_t* packed;         /* HOST [E] out: state bits [N-1:0] | terminated << 30 | truncated << 31.  The reward is a
                               function of (number of distinct non-zero actions of the env, terminated): the caller
                               looks it up in pbn_reward_table instead of moving 4 more bytes per env */
  const uint16_t* actions16; /* HOST [E] in, instead of `actions`: a0 | a1 << 5 | a2 << 10 (each action 0..N <= 30) */
  uint16_t* actions16_dev;  /* DEVICE [E] staging buffer for actions16, caller-owned (actions_dev is needed as well) */
} pbn_host_io;

/* env.step(action) with HOST buffers, end to end: copies the actions to the device, steps all
 * n_envs instances (exactly as pbn_step with args->actions = io->actions_dev) and copies the
 * results back.  The batch is cut into lanes, ranges of whole 1024-env tiles; each lane runs action
 * upload -> step -> result download in order on its own library stream, and the lanes run
 * concurrently, so one lane's upload overlaps another lane's download.  n_chunks sets the number of
 * lanes (at most 16 and the number of tiles); 0 picks 1 below 2^18 envs, else 2, or 4 for the
 * graph-replayed calls below.  Envs are independent, so the result does not depend on the number of
 * lanes.  Unlike the device entry points this call BLOCKS until the host outputs are complete (like
 * the reference's env.step it returns values); it waits on its own streams only, never on the whole
 * device, and later work on `stream` is ordered after the step.
 * The lanes share one counter value.  With args->step_ctr_dev set and neither PBN_STEP_PDL nor PBN_STEP_NO_COUNT,
 * the call adds 1 to *step_ctr_dev itself once the lanes have joined, so its arguments can stay the same from call to
 * call.  When only `packed` is requested, with actions16 and args->step_ctr_dev set, the library captures the whole
 * step the second time it sees an (args, io) pair and replays it as one CUDA graph launch afterwards (8 pairs are kept;
 * keep the buffers alive while the handle may still replay them). */
int pbn_step_host(pbn_handle* h, const pbn_step_args* args, const pbn_host_io* io, void* stream);

/* reward = table[n_flips + (bins + 1) * terminated], n_flips = number of distinct action values in 1..N of the env
 * (the fp32 values pbn_step writes): out[2 * (bins + 1)] (HOST). */
int pbn_reward_table(const pbn_handle* h, float* out, int32_t n);

/* ---- Plane-resident env state (sliced kernel) -----------------------------------------------------------
 * The env state an agent never looks at between steps -- packed states, target ids, episode counters -- can
 * live on the device in the layout the bit-sliced kernel computes in (bit-planes over tiles of 1024 envs,
 * csrc/step_planes.cuh), so that a step neither transposes nor touches per-env state words: pbn_step with
 * args->resident set is the fastest form of env.step (bdq_model/__init__.py:177).  The row-format arrays of
 * pbn_step_args stay the boundary format: pbn_resident_import builds the block from them (state words,
 * target ids -- negative or >= min(A, 255) = no target --, counters; needs the attractor table for the
 * target planes, so call it after pbn_update_attractors), pbn_resident_export writes them back (any output
 * may be NULL).  Results are bit-identical to pbn_step on the row-format arrays (same random streams).
 * Supported: networks the sliced kernel takes, at most 254 attractors, and either single-state attractors
 * without wildcards (any number) or attractor tables of at most 256 (care, value) entries.
 * pbn_resident_words: size of the block in 32-bit words (whole tiles + one epoch word per tile for
 * PBN_STEP_CHAIN; 128-byte aligned memory). */
int64_t pbn_resident_words(const pbn_handle* h, int64_t n_envs);
int pbn_resident_import(pbn_handle* h, uint32_t* resident, const uint64_t* state, const int32_t* target_id,
                        const uint16_t* t, int64_t n_envs, void* stream);
int pbn_resident_export(pbn_handle* h, const uint32_t* resident, uint64_t* state, int32_t* target_id,
                        uint16_t* t, int64_t n_envs, void* stream);

/* n_steps uncontrolled network updates of every instance in ONE launch (env.step([]) n_steps times,
 * graph_classifier/__init__.py:148; the burn-in of the attractor search; the long runs of compute_ssd_hist,
 * train_pbn_28.py:257): the states are loaded once, stay on chip as bit-planes between updates and are
 * written back once.  Bit-identical to n_steps calls of pbn_step with actions = NULL and step counters
 * step_ctr .. step_ctr + n_steps - 1 as far as `state` is concerned; t / target / reward / flags are not
 * touched, nothing is reset.  stats (DEVICE, may be NULL): PBN_STAT_STEPS and PBN_STAT_PERTURBED are
 * accumulated.  Sliced kernel only (PBN_ERR_UNSUPPORTED otherwise: loop over pbn_step instead). */
int pbn_rollout(pbn_handle* h, uint64_t* state, int64_t n_steps, uint64_t step_ctr, int64_t env_offset,
                int64_t n_envs, unsigned long long* stats, void* stream);

/* ---- Steady-state statistics (compute_ssd_hist, train_pbn_28.py:257) ---------------------------------------
 * A record ADDS into caller-owned DEVICE u64 accumulators and never overwrites them, so successive calls and shards
 * of a batch can be summed:
 *   gene_on [N] (may be NULL): gene_on[g] += the number of recorded env-states in which gene g is 1;
 *   hist [2^n_proj] (may be NULL): the states projected onto the n_proj (0..12) distinct genes proj_genes[0..n_proj)
 *     (a HOST array): bin b = sum_j bit(state, proj_genes[j]) << j (the packing of steady_state_histogram(genes=...));
 *     with n_proj = 0, hist[0] counts every recorded state.
 * Only real envs are counted, never the padding of a ragged last tile.  Invalid input (n_proj > 12, a repeated or
 * out-of-range projection gene, stride < 1, the pbn_rollout checks) returns PBN_ERR_INVALID. */
/* n_steps uncontrolled updates exactly as pbn_rollout (same streams, same final states, same stats), and after
 * update s (s = 1..n_steps) the states are recorded iff s % stride == 0.  Sliced kernel only (PBN_ERR_UNSUPPORTED
 * otherwise).  The recording kernel is a separate specialisation, compiled on the first call. */
int pbn_rollout_record(pbn_handle* h, uint64_t* state, int64_t n_steps, uint64_t step_ctr, int64_t env_offset,
                       int64_t n_envs, int32_t stride, const int32_t* proj_genes, int32_t n_proj,
                       unsigned long long* gene_on, unsigned long long* hist, unsigned long long* stats, void* stream);
/* Record n_envs row-format states once (any kernel): after a pbn_step, for policy-in-the-loop statistics. */
int pbn_record_states(pbn_handle* h, const uint64_t* state, int64_t n_envs, const int32_t* proj_genes,
                      int32_t n_proj, unsigned long long* gene_on, unsigned long long* hist, void* stream);

/* The same step with injected predictor choices / perturbation masks: the parity entry point
 * (deterministic core T of SURVEY.md 8a-4).  args->sel must be non-NULL. */
int pbn_step_injected(pbn_handle* h, const pbn_step_args* args, void* stream);

/* env.reset() (bdq_model/__init__.py:161,204): for envs with done_mask[e] != 0 (all if NULL)
 * draw (source, target) from the pair table, set state to a random state of the source
 * attractor ('*' -> 0, model_tester.py:609), t = 0. */
int pbn_reset(pbn_handle* h, uint64_t* state, int32_t* target_id, int32_t* source_id, uint16_t* t,
              const uint8_t* done_mask, uint64_t step_ctr, int64_t env_offset, int64_t n_envs,
              void* stream);

/* env.render() / observation for the agent (bdq_model/__init__.py:92): packed words ->
 * [E,N] uint8 or float32. */
int pbn_unpack(pbn_handle* h, const uint64_t* state, void* out, int32_t out_kind, int64_t n_envs,
               void* stream);

/* Inverse of pbn_unpack: [E,N] uint8 -> packed words (env.graph.setState, model_tester.py:611). */
int pbn_pack(pbn_handle* h, const uint8_t* bits, uint64_t* state, int64_t n_envs, void* stream);

/* env.is_attracting_state / state_attractor_id: index of the first attractor containing each
 * state, -1 if none (graph_classifier/__init__.py:129-134; bdq_model/__init__.py:180). */
int pbn_attractor_id(pbn_handle* h, const uint64_t* state, int32_t* attr_id, int64_t n_envs,
                     void* stream);

/* ---- Device-resident replay ring + fused observation unpack (the callers' side of the path) ----------
 * Replaces the python-list ExperienceReplay (bdq_model/memory.py:22-70: store / sample) and the tuple ->
 * float-tensor rebuilds of predict() and update_policy() (bdq_model/__init__.py:92-93,100-109).
 * Transitions stay packed; all arrays are caller-owned DEVICE memory holding `capacity` transitions. */
typedef struct {
  uint64_t* state;       /* [capacity*W] state the action was chosen in */
  uint64_t* next_state;  /* [capacity*W] state after the step (before any auto-reset) */
  int32_t* target_id;    /* [capacity]   target attractor of the episode */
  uint8_t* actions;      /* [capacity*bins] */
  float* reward;         /* [capacity] */
  uint8_t* done;         /* [capacity]   terminated | truncated << 1 */
  int64_t capacity;
} pbn_replay;

/* memory.store(), first half, BEFORE the step: ring slot (head + e) mod capacity <- (state[e], target_id[e]). */
int pbn_replay_observe(pbn_handle* h, const pbn_replay* r, int64_t head, const uint64_t* state,
                       const int32_t* target_id, int64_t n_envs, void* stream);
/* memory.store(), second half, AFTER the step: the same slots <- (actions, reward, done flags, next_state);
 * pass the step's final_state as next_state when auto-reset is on.  actions/truncated may be NULL. */
int pbn_replay_commit(pbn_handle* h, const pbn_replay* r, int64_t head, const uint8_t* actions, const float* reward,
                      const uint8_t* terminated, const uint8_t* truncated, const uint64_t* next_state,
                      int64_t n_envs, void* stream);
/* memory.sample() + the tensor building of update_policy(): for ring slots index[0..B) (DEVICE int64) write
 * obs [2,B,N] = (state bits, target-state bits), next_obs [2,B,N] = (next-state bits, target-state bits) as
 * float32, actions [B,bins] int64, reward [B], done [B] float32 (1.0 if terminated or truncated).  Any output
 * may be NULL.  The target state is the first state of the attractor with '*' -> 0 (env.reset()'s `target`). */
int pbn_replay_sample(pbn_handle* h, const pbn_replay* r, const int64_t* index, int64_t batch, float* obs,
                      float* next_obs, int64_t* actions, float* reward, float* done, void* stream);
/* ---- Prioritised replay over the ring's slots (proportional PER, Schaul et al.; the sum / min segment trees of
 * the reference's data_structures.py and ddqn_per/, SURVEY.md section 2 rows 13-14, in the form of OpenAI baselines).
 * Parity with the reference is not pinned (its tests are stale); this contract is the project's own.
 *
 * Layout.  L = the smallest power of two >= capacity, D = log2 L.  `tree` holds pbn_per_tree_floats(capacity) = 5L
 * words of caller-owned DEVICE memory, every binary level of both trees stored as a heap (node k has children 2k and
 * 2k+1, the root is node 1, leaf of slot i is node L + i):
 *   tree[k]            k in [1, 2L)  sum tree S: leaves p[i] (fp32), S(node) = S(2 node) + S(2 node + 1), one fp32 add
 *                                    with round-to-nearest; total = tree[1]
 *   tree[2L + k]       k in [1, 2L)  min tree M: the same shape built with fminf; pmin = tree[2L + 1]
 *   tree[0]                          scratch of the kernels (a completion ticket, zero between calls)
 *   tree[4L .. 5L)                   scratch of the kernels (int32 owner per leaf, -1 between calls)
 * Unwritten leaves are 0 in S and +inf in M.  max_p (DEVICE, one float) is the largest raw priority seen, 1.0
 * initially.  pbn_per_init establishes this state; nothing else may write the arrays.
 *
 * push(head, n), after pbn_replay_commit with the same head: slots (head + e) mod capacity, e < n, get the leaf
 *   powf(max_p, alpha), and all their ancestors are rebuilt.
 * update(index[B], td[B], eps): raw = fminf(fmaxf(fabsf(td), 0) + eps, 1e30f) (NaN -> eps, +-inf -> 1e30, so the
 *   trees never hold NaN or inf); the leaf becomes powf(raw, alpha); max_p = max(max_p, raw) over the valid entries.
 *   When a slot occurs more than once the LAST occurrence in batch order wins.  Indices outside [0, capacity) are
 *   ignored (a device-side index cannot be validated without a synchronisation).  eps > 0.
 * sample(u[B], beta) -> index[B] (int64), weight[B] (fp32); u in [0, 1) fp32 from the caller, B <= 2^24:
 *   seg = total / B; mass_b = fl(fl(u_b * seg) + fl(b * seg)) (no FMA); descent from the root: go left if
 *   left > mass or right == 0, else mass = fl(mass - left) and go right -- every visited node has a positive sum,
 *   so the result is a written slot; weight_b = powf(pmin / p[index_b], beta), which is baselines'
 *   (P * size)^-beta / max_w with size and total cancelled: no host-side size, so the call can be captured in a
 *   CUDA graph (with beta frozen into it).
 * All calls run on the caller's stream without synchronising; calls on one tree must be ordered on one stream.
 * alpha >= 0 and beta >= 0, finite; capacity <= 2^30. */
typedef struct {
  float* tree;           /* [pbn_per_tree_floats(capacity)] sum tree, min tree and scratch (layout above) */
  float* max_p;          /* [1] largest raw priority so far */
  int64_t capacity;      /* slots of the replay ring the trees index */
  float alpha;           /* priority exponent */
  float reserved;
} pbn_per;

/* Words of the tree array for a ring of `capacity` slots (5 * L), or a negative status. */
int64_t pbn_per_tree_floats(int64_t capacity);
/* Empty trees (S = 0, M = +inf), max_p = 1.0, scratch cleared. */
int pbn_per_init(pbn_handle* h, const pbn_per* p, void* stream);
/* New transitions enter at the running maximum priority. */
int pbn_per_push(pbn_handle* h, const pbn_per* p, int64_t head, int64_t n, void* stream);
/* New priorities from TD errors for ring slots index[0..B) (DEVICE int64 / fp32). */
int pbn_per_update(pbn_handle* h, const pbn_per* p, const int64_t* index, const float* td_error, int64_t batch,
                   float eps, void* stream);
/* Stratified proportional sample of B slots and their importance weights (DEVICE arrays). */
int pbn_per_sample(pbn_handle* h, const pbn_per* p, const float* u, int64_t batch, float beta, int64_t* index,
                   float* weight, void* stream);

/* The agent's network input for the live envs (predict(), bdq_model/__init__.py:92-93):
 * obs [2,E,N] float32 = (state bits, target-state bits). */
int pbn_observe(pbn_handle* h, const uint64_t* state, const int32_t* target_id, float* obs, int64_t n_envs,
                void* stream);

/* ---- Batched all-pairs evaluation (model_tester.py:584-658) -------------------------------------------
 * E rollouts (run x source attractor x target attractor) are stepped together with pbn_step; these entry
 * points do the reference loop's bookkeeping on the device. */
/* env.in_target(state) for every instance (model_tester.py:616): out[e] = 1 iff state[e] is in attractor
 * target_id[e]. */
int pbn_in_target(pbn_handle* h, const uint64_t* state, const int32_t* target_id, uint8_t* out, int64_t n_envs,
                  void* stream);
/* After a step, for rollouts with active[e] != 0: count[e] += 1; if count[e] > max_steps the rollout has failed
 * (model_tester.py:627-636 books max_steps + 1 = 101) and stops; else if terminated[e] it stops with count[e]
 * steps.  n_active (DEVICE, may be NULL) is incremented by the number of rollouts still running. */
int pbn_rollout_track(pbn_handle* h, const uint8_t* terminated, uint8_t* active, int32_t* count,
                      int32_t max_steps, int64_t n_envs, unsigned int* n_active, void* stream);
/* result_matrix[pair] += count, data[count] += 1 (model_tester.py:645-652): matrix [n_pairs] and
 * hist [max_steps + 2] are DEVICE u64 accumulators; pair_id[e] = source * A + target. */
int pbn_rollout_reduce(pbn_handle* h, const int32_t* count, const int32_t* pair_id, int64_t n_envs,
                       int32_t n_pairs, int32_t max_steps, unsigned long long* matrix,
                       unsigned long long* hist, void* stream);

/* ---- Attractor discovery / steady-state statistics (print_graph.py:15-34, train_pbn_28.py:257) -------
 * Visit-count hash table in DEVICE memory: tags[capacity] (0 = empty slot), slot_state[capacity*W],
 * counts[capacity], capacity a power of two, all zero-initialised by the caller.  For every instance with
 * mask[e] != 0 (all if mask is NULL) counts[slot of state[e]] += 1; *overflow (DEVICE) counts states
 * that found no slot (table too full).  tags[] holds 2*state+1 for N <= 63 and a splitmix64 fingerprint
 * otherwise (csrc/discover.cuh); a fingerprint match is confirmed against slot_state, so distinct states never
 * merge.  The value 1 marks a slot whose state words are being published. */
int pbn_visit_count(pbn_handle* h, const uint64_t* state, const uint8_t* mask, int64_t n_envs,
                    unsigned long long* tags, uint64_t* slot_state, unsigned long long* counts,
                    int64_t capacity, unsigned int* overflow, void* stream);
/* Successor descriptor of the perturbation-free state-transition graph (graph.genSTG(), print_graph.py:15-21)
 * for a list of states: bit i of can1[e] / can0[e] = some predictor of gene i yields 1 / 0 in state[e].
 * The successors of state[e] are {t : t_i = 1 where only can1, 0 where only can0, free where both}. */
int pbn_successor_sets(pbn_handle* h, const uint64_t* state, int64_t n_states, uint64_t* can1, uint64_t* can0,
                       void* stream);

/* Exact attractors of large networks: forward closure of a candidate state and backward reachability, on
 * the device.  `list` [list_cap*W] holds the closure in discovery order (the caller writes the seed into
 * list[0], sets *list_count = 1 and registers it in the table with index 1); the hash table is the
 * visit-count table above with its counts column reused as slot_index = list index + 1.
 * pbn_closure_expand appends every successor of list[begin, end) that is not in the table yet;
 * *status (DEVICE int) becomes 1 if a state has more than max_free free genes (2^max_free successors),
 * 2 if the list is full, 3 if the table is full.  pbn_closure_reach does one sweep of "flags[i] = 1 if a
 * successor of list[i] has flag 1" and sets *changed (DEVICE int) if any flag changed. */
int pbn_closure_expand(pbn_handle* h, uint64_t* list, int64_t begin, int64_t end, int64_t list_cap,
                       unsigned long long* list_count, unsigned long long* tags, uint64_t* slot_state,
                       unsigned long long* slot_index, int64_t capacity, int32_t max_free, int32_t* status,
                       void* stream);
int pbn_closure_reach(pbn_handle* h, const uint64_t* list, int64_t count, uint8_t* flags,
                      const unsigned long long* tags, const uint64_t* slot_state,
                      const unsigned long long* slot_index, int64_t capacity, int32_t* changed, void* stream);

/* ---- Exhaustive attractor search: backward reachability over every state (N <= PBN_REACH_MAX_GENES) -------------
 * Without perturbation every state reaches an attractor (a sink SCC of the STG above) and attractors are closed.  So
 * mark the states of the attractors found so far (pbn_reach_mark) and repeat pbn_reach_sweep -- "mark s if some
 * successor of s is marked" -- until a sweep marks nothing: if every state is then marked, no other attractor exists;
 * otherwise the unmarked states are closed under successors and hold at least one attractor not found yet.  The fixed
 * point is the set of states that reach a marked seed; it does not depend on the order of the marks within a sweep
 * (csrc/discover.cuh).  Both calls run on the caller's stream without synchronising or allocating, in launches of at
 * most 2^22 states.
 * marks: DEVICE uint32 [max(1, 2^N / 32)], bit (s & 31) of word s >> 5 = state s.  *newly (DEVICE u64) is
 * increased by the number of bits the call set.  Perturbation-free STG whatever the handle's perturb_p.
 * N > PBN_REACH_MAX_GENES: PBN_ERR_UNSUPPORTED; NULL marks / newly: PBN_ERR_INVALID.
 * The limit is not the DP's: the bitset needs one bit per state (2 GiB at 34 genes). */
#define PBN_REACH_MAX_GENES 34
/* Set the bits of states[0, n_states) (DEVICE u64, one index per state); states >= 2^N are ignored. */
int pbn_reach_mark(pbn_handle* h, uint32_t* marks, const uint64_t* states, int64_t n_states,
                   unsigned long long* newly, void* stream);
/* One sweep over every unmarked state. */
int pbn_reach_sweep(pbn_handle* h, uint32_t* marks, unsigned long long* newly, void* stream);
/* Forward closure: one sweep that expands every state of `set` not yet in `done` (both DEVICE uint32 bitsets in the
 * marks layout): the bits of all its successors are set in `set`, and the state's bit in `done`.  Repeated until a
 * sweep expands nothing, `set` is the forward closure of its initial bits and `done` equals it.  newly: DEVICE u64 [2],
 * increased by the number of bits set in `set` and by the number of states expanded.  Bitsets of 2^N / 8 bytes, one
 * bit per state, whatever the closure's size or its states' free genes.  Same refusals as pbn_reach_sweep (NULL
 * done: PBN_ERR_INVALID). */
int pbn_reach_forward(pbn_handle* h, uint32_t* set, uint32_t* done, unsigned long long* newly, void* stream);

/* ---- Exact optimal control: finite-horizon dynamic programming over every state (N <= PBN_DP_MAX_GENES) ----------
 * The env is a finite Markov decision process, so for networks whose 2^N states fit on the GPU the best possible policy
 * of a target can be computed exactly by backward induction -- the yardstick an agent's strategy lengths and returns are
 * compared against.  States are indices s in [0, 2^N) (bit i = gene i); a flip mask m is a subset of the controllable
 * genes with popcount(m) <= max_flips; one env step from s with mask m starts from u = s ^ m and draws t ~ P(u -> .),
 * P = items 2-4 of "One env step" above with the handle's perturbation model and perturb_p.  A backup is
 *   W = P U (pbn_dp_expect),   V(s) = max_m fl(r_action |m|) + W[s ^ m] (pbn_dp_improve),
 * the rest (rewards, discount, target and wrong-attractor terms) is elementwise work of the caller
 * (pbn_rl_b200/control.py).  Perturbation: NONE: P = F (the selection step); B: P = F K_p; A: P = (1-p)^N F +
 * K_p - (1-p)^N I, K_p = the per-gene binary symmetric channel (a perturbed step skips the update and lands on
 * u ^ pert, pert != 0); model C with p > 0 makes nearly every gene free in every state (a backup of O(4^N)) and is
 * refused; any model with p = 0 is NONE.
 * The exact state distribution after a step, x P, is pbn_dp_push.  All three calls run on the caller's stream without
 * synchronising or allocating, in launches of at most 2^22 states, and are deterministic: the same inputs give
 * bit-identical outputs (no floating-point atomics). */
#define PBN_DP_MAX_GENES 28
/* Bytes of caller-owned DEVICE workspace the three calls below need for this handle (24 * 2^N), or a negative status:
 * PBN_ERR_UNSUPPORTED when N > PBN_DP_MAX_GENES or the perturbation model is C with p > 0. */
int64_t pbn_dp_workspace_bytes(const pbn_handle* h);
/* w[u] = sum_t P(u -> t) u_in[t] for every u in [0, 2^N)  (fp64, DEVICE arrays of 2^N; w must not alias u_in).  P: one
 * step of the handle's dynamics without interventions -- predictor selection with probabilities func_prob (DEVICE fp64
 * [F], the network's selection probabilities in func_offset order; not validated), then the handle's perturbation model
 * at perturb_p.  workspace: pbn_dp_workspace_bytes (may be NULL when p = 0). */
int pbn_dp_expect(pbn_handle* h, const double* func_prob, const double* u_in, double* w, void* workspace, void* stream);
/* v[s] = max over masks m with m subset of flip_genes and popcount(m) <= max_flips of  fl(r_action * popcount(m)) +
 * w[s ^ m] (no FMA); policy[s] = that m (may be NULL).  Ties: fewer flips, then larger w[s ^ m], then smaller s ^ m.
 * r_action <= 0, 0 <= max_flips <= PBN_MAX_BINS, flip_genes within the N genes, else PBN_ERR_INVALID.  v must not alias
 * w; workspace (pbn_dp_workspace_bytes) may be NULL when max_flips <= 1. */
int pbn_dp_improve(pbn_handle* h, const double* w, uint64_t flip_genes, int32_t max_flips, double r_action,
                   double* v, uint32_t* policy, void* workspace, void* stream);
/* y = x P (masks == NULL) or x P_mu, P_mu(s, .) = P(s ^ masks[s], .) -- the forward operator of pbn_dp_expect, for
 * state distributions: y[t] = sum_s x_in[s] P_mu(s -> t), one env step from distribution x_in with the flips
 * masks[s] (DEVICE uint32 [2^N], bits at gene N and above ignored; NULL: no interventions) applied first.  x_in, y:
 * DEVICE fp64 [2^N], y must not alias x_in; func_prob as for pbn_dp_expect; workspace: pbn_dp_workspace_bytes (may be
 * NULL when p = 0 and masks == NULL).  The sums are exact integer sums in fixed point: every term x_in[s] P(s -> t) of
 * the selection step (and x_in[s] of the interventions) is rounded to the nearest multiple of 2^-63, losing at most
 * 2^-64, so y is bit-identical from call to call whatever the order of the additions.  This needs x_in >= 0 and
 * sum x_in <= 1 (a probability or sub-probability vector; not validated).  Perturbation is applied in fp64 after the
 * selection step (model B) or mixed in with c = (1-p)^N (model A: y = c x F + x K_p - c x). */
int pbn_dp_push(pbn_handle* h, const double* func_prob, const double* x_in, const uint32_t* masks, double* y,
                void* workspace, void* stream);

/* *step_ctr_dev += n on the stream (fully serialised): closes a sequence of PBN_STEP_PDL launches. */
int pbn_advance_counter(pbn_handle* h, uint64_t* step_ctr_dev, uint64_t n, void* stream);

/* Introspection. */
/* Slots of the hash set pbn_update_attractors built over the fully specified attractor states (tables with an
 * attractor of more than 64 states: env.in_target / env.is_attracting_state become one probe sequence, model_tester.py:
 * 602-616), 0 if the table is small enough for the scan. */
int pbn_attractor_hash_slots(const pbn_handle* h);
int pbn_kernel_kind(const pbn_handle* h);            /* PBN_KERNEL_SCALAR or PBN_KERNEL_SLICED */
int pbn_words_per_state(const pbn_handle* h);        /* W */
int pbn_launch_count(const pbn_handle* h, uint64_t* out); /* kernels launched through this handle */

/* Load-time specialisation.  pbn_jit_source writes the CUDA source generated for this network
 * (the predictor functions as LOP3 trees + selection logic, net_gen.cuh / net_update.inc) into
 * buf (NUL-terminated, truncated to len) and returns the full length, or a negative status if
 * the network is not eligible for the sliced kernel.  pbn_jit_precompile compiles that
 * specialisation with NVRTC for sm_100a into the on-disk cache (no GPU needed), so that a later
 * pbn_create on the GPU box only loads the cubin. */
int64_t pbn_jit_source(const pbn_net_desc* desc, int injected, char* buf, int64_t len);
int pbn_jit_precompile(const pbn_net_desc* desc);
const char* pbn_last_error(void);
const char* pbn_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PBN_B200_H */
