// C-ABI of libpbn_b200.so (include/pbn_b200.h): handle management, table upload, launches.
// The only translation unit; kernels live in the .cuh files next to it.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <new>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "pbn_common.cuh"
#include "step_scalar.cuh"
#include "sliced_host.cuh"
#include "replay.cuh"
#include "evaluate.cuh"
#include "discover.cuh"
#include "resident.cuh"
#include "per.cuh"
#include "record.cuh"
#include "control.cuh"

using namespace pbn;

namespace {

thread_local char g_err[512] = "";
// The handle whose pbn_advance_counter was the last launch made through the library (else null): the next step of
// THAT handle must not start before the counter update is complete and visible, so it is launched without the
// programmatic-serialisation attribute.  Any other launch in between is itself fully serialised behind the update.
const void* g_last_advance = nullptr;

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define PBN_CUDA(expr)                                                                      \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess)                                                                  \
      return fail(PBN_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess) ok = true;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

template <typename T>
int upload(T** dptr, const T* host, size_t count, cudaStream_t stream = nullptr) {
  if (*dptr) {
    cudaFree(*dptr);
    *dptr = nullptr;
  }
  if (count == 0) return PBN_OK;
  PBN_CUDA(cudaMalloc(reinterpret_cast<void**>(dptr), count * sizeof(T)));
  PBN_CUDA(cudaMemcpyAsync(*dptr, host, count * sizeof(T), cudaMemcpyHostToDevice, stream));
  PBN_CUDA(cudaStreamSynchronize(stream));  // host buffers are the caller's temporaries
  return PBN_OK;
}

// Device table with spare capacity: updated in place on the caller's stream, reallocated (after a stream
// synchronisation) only when it outgrows its capacity -- so pointers captured in CUDA graphs stay valid.
template <typename T>
int update_table(T** dptr, size_t* cap, const T* host, size_t count, cudaStream_t stream) {
  if (count > *cap) {
    PBN_CUDA(cudaStreamSynchronize(stream));  // kernels in flight may still read the old allocation
    size_t ncap = *cap ? *cap : 64;
    while (ncap < count) ncap *= 2;
    if (*dptr) cudaFree(*dptr);
    *dptr = nullptr;
    *cap = 0;
    PBN_CUDA(cudaMalloc(reinterpret_cast<void**>(dptr), ncap * sizeof(T)));
    *cap = ncap;
  }
  if (count) PBN_CUDA(cudaMemcpyAsync(*dptr, host, count * sizeof(T), cudaMemcpyHostToDevice, stream));  // pageable source: staged before the call returns
  return PBN_OK;
}

}  // namespace

struct pbn_handle {
  int device = 0;
  int W = 1;
  int kernel = PBN_KERNEL_SCALAR;
  int num_sms = 148;
  double perturb_p = 0.0;   // the perturbation probability as given (exact control needs it in fp64)
  NetParams net{};
  // owned device tables
  int32_t* d_func_offset = nullptr;
  FuncDesc* d_funcs = nullptr;
  uint32_t* d_func_cum = nullptr;
  uint32_t* d_survival = nullptr;
  int32_t* d_attr_offset = nullptr;
  uint64_t* d_attr_care = nullptr;
  uint64_t* d_attr_val = nullptr;
  uint32_t* d_pair_cum = nullptr;
  size_t cap_attr_offset = 0, cap_attr_care = 0, cap_attr_val = 0, cap_pair_cum = 0;
  // hash set over the fully specified attractor states + CSR of the wildcard entries (large attractors)
  unsigned long long* d_ahash_tags = nullptr;
  uint64_t* d_ahash_state = nullptr;
  int32_t* d_ahash_attr = nullptr;
  int32_t* d_awild_offset = nullptr;
  int32_t* d_awild_entry = nullptr;
  size_t cap_ahash_tags = 0, cap_ahash_state = 0, cap_ahash_attr = 0, cap_awild_offset = 0, cap_awild_entry = 0;
  unsigned int* d_ticket = nullptr;
  uint32_t* d_surv_sliced = nullptr;
  WideDesc* d_wide = nullptr;
  uint64_t* d_wide_lut = nullptr;
  // sliced kernel: the network's JIT programs (kJitParts), [part][0 = own-RNG, 1 = injected randomness], each loaded
  // on first use
  jit::GenNet gen;
  struct JitKernel {
    cudaKernel_t k = nullptr;
    uint32_t smem_opt_in = 48u * 1024u;   // ensure_dynamic_smem's cache
  };
  struct JitProgram {
    cudaLibrary_t lib = nullptr;
    std::string key;         // shared-module registry key (release_module)
    JitKernel kernel[3];     // in the order of kJitParts[part].kernels
  };
  JitProgram jit[3][2];
  std::vector<uint32_t> surv_sliced_host;  // copied into every loaded specialisation's constant memory
  int sliced_threads = 128, sliced_min_blocks = 1;
  uint32_t scalar_smem_opt_in = 48u * 1024u;   // step_scalar_kernel (one instance per handle)
  uint64_t launches = 0;
  // pbn_step_host: one stream and one join event per lane (created on first use)
  static constexpr int kMaxLanes = 16;
  cudaStream_t s_lane[kMaxLanes] = {};
  cudaEvent_t ev_k[kMaxLanes] = {};
  // packed form with a device step counter: the whole step (uploads, unpack, step, export kernels of all lanes, counter
  // update) is captured once per distinct argument set and replayed as one CUDA graph launch afterwards
  struct HostGraph {
    pbn_step_args a;
    pbn_host_io io;
    int seen = 0;
    uint64_t launches = 0, last_use = 0;
    cudaGraphExec_t exec = nullptr;
  };
  static constexpr int kHostGraphs = 8;
  HostGraph host_graph[kHostGraphs];
  uint64_t host_graph_clock = 0;
  cudaStream_t s_origin = nullptr;
  cudaEvent_t ev_entry = nullptr, ev_fork = nullptr, ev_done = nullptr;
};

// Loaded specialisations are shared between the handles of a process: env batches of the same network (the bench
// rotates eight of them, an RL loop holds a train and an eval batch) then launch ONE copy of the kernel code, which
// stays warm in the instruction caches, instead of one copy per handle.  A module is identified by its cubin and by the
// survival table its constant memory holds (handles with another perturbation rate get their own).
struct SharedModule {
  cudaLibrary_t lib = nullptr;
  int refs = 0;
};
static std::mutex g_modules_mutex;
static std::map<std::string, SharedModule> g_modules;

static uint64_t fnv1a(const void* data, size_t n, uint64_t hsh = 1469598103934665603ull) {
  const unsigned char* p = static_cast<const unsigned char*>(data);
  for (size_t i = 0; i < n; ++i) hsh = (hsh ^ p[i]) * 1099511628211ull;
  return hsh;
}

// returns the module (loading it and filling its survival table on first use) and the key to release it with
static int acquire_module(pbn_handle* h, const std::vector<char>& cubin, bool own_rng, cudaLibrary_t* lib, std::string* key) {
  uint64_t a = fnv1a(cubin.data(), cubin.size());
  uint64_t b = own_rng ? fnv1a(h->surv_sliced_host.data(), h->surv_sliced_host.size() * sizeof(uint32_t)) : 0ull;
  char buf[96];
  snprintf(buf, sizeof(buf), "%d:%zu:%016llx:%016llx", h->device, cubin.size(), (unsigned long long)a, (unsigned long long)b);
  std::lock_guard<std::mutex> lock(g_modules_mutex);
  SharedModule& m = g_modules[buf];
  if (!m.lib) {
    cudaLibrary_t l = nullptr;
    const cudaError_t e = cudaLibraryLoadData(&l, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (e != cudaSuccess) {
      g_modules.erase(buf);
      return fail(PBN_ERR_CUDA, "cudaLibraryLoadData: %s", cudaGetErrorString(e));
    }
    if (own_rng) {  // the survival table of the perturbation sub-streams lives in the specialisation's constant memory
      void* dptr = nullptr;
      size_t bytes = 0;
      cudaError_t e2 = cudaLibraryGetGlobal(&dptr, &bytes, l, "_ZN3pbn10kSurvTableE");
      if (e2 == cudaSuccess && bytes != h->surv_sliced_host.size() * sizeof(uint32_t)) e2 = cudaErrorInvalidValue;
      if (e2 == cudaSuccess) e2 = cudaMemcpy(dptr, h->surv_sliced_host.data(), bytes, cudaMemcpyHostToDevice);
      if (e2 != cudaSuccess) {
        cudaLibraryUnload(l);
        g_modules.erase(buf);
        return fail(PBN_ERR_JIT, "kSurvTable of the specialisation: %s (%zu bytes, expected %zu)", cudaGetErrorString(e2), bytes,
                    h->surv_sliced_host.size() * sizeof(uint32_t));
      }
    }
    m.lib = l;
  }
  m.refs += 1;
  *lib = m.lib;
  *key = buf;
  return PBN_OK;
}

static void release_module(const std::string& key) {
  if (key.empty()) return;
  std::lock_guard<std::mutex> lock(g_modules_mutex);
  auto it = g_modules.find(key);
  if (it == g_modules.end()) return;
  if (--it->second.refs <= 0) {
    cudaLibraryUnload(it->second.lib);
    g_modules.erase(it);
  }
}

// Dynamic shared memory above 48 KB must be opted into per kernel -- and the kernels are shared between handles, so the
// handle's cached value is only a shortcut: the kernel's own attribute decides, and it is only ever raised.
static int ensure_dynamic_smem(const void* k, uint32_t bytes, uint32_t* cached) {
  if (bytes <= *cached) return PBN_OK;
  cudaFuncAttributes fa{};
  PBN_CUDA(cudaFuncGetAttributes(&fa, k));
  uint32_t cur = fa.maxDynamicSharedSizeBytes > 0 ? (uint32_t)fa.maxDynamicSharedSizeBytes : 0u;
  if (cur < 48u * 1024u) cur = 48u * 1024u;
  if (bytes > cur) {
    PBN_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    cur = bytes;
  }
  *cached = cur;
  return PBN_OK;
}

// Every kernel launch of the library goes through launch(), which counts it (pbn_launch_count) and applies the PDL
// rule: a step launched with PBN_STEP_PDL reads *step_ctr_dev before its griddepcontrol.wait, and a primary grid's
// writes are only guaranteed visible after the wait, so when the launch right before it is this handle's own
// pbn_advance_counter, the step is launched fully serialised instead.
template <typename Go>
static int launch_with(pbn_handle* h, const void* k, unsigned grid, unsigned block, uint32_t smem, cudaStream_t stream,
                       bool pdl, Go go) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  if (pdl && g_last_advance != h) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  const cudaError_t e = go(&cfg);
  if (e != cudaSuccess) {
    const char* name = nullptr;
    if (cudaFuncGetName(&name, k) != cudaSuccess || !name) name = "kernel";
    cudaGetLastError();   // the error is returned here; a later check must not see it again
    return fail(PBN_ERR_CUDA, "launch of %s (grid %u, block %u, %u B shared memory) failed: %s", name, grid, block, smem,
                cudaGetErrorString(e));
  }
  h->launches += 1;
  g_last_advance = nullptr;
  return PBN_OK;
}

// A kernel of this library: the arguments are converted to the kernel's parameter types.
template <typename... P, typename... A>
static int launch(pbn_handle* h, void (*k)(P...), unsigned grid, unsigned block, uint32_t smem, cudaStream_t stream,
                  bool pdl, A&&... args) {
  return launch_with(h, reinterpret_cast<const void*>(k), grid, block, smem, stream, pdl,
                     [&](const cudaLaunchConfig_t* cfg) { return cudaLaunchKernelEx(cfg, k, std::forward<A>(args)...); });
}

// A kernel of a JIT program.
static int launch(pbn_handle* h, cudaKernel_t k, unsigned grid, unsigned block, uint32_t smem, cudaStream_t stream,
                  bool pdl, void** args) {
  const void* f = reinterpret_cast<const void*>(k);
  return launch_with(h, f, grid, block, smem, stream, pdl,
                     [&](const cudaLaunchConfig_t* cfg) { return cudaLaunchKernelExC(cfg, f, args); });
}

// The JIT programs of a network (jit::compile's `part`) and the kernels each one holds: [0] the own-RNG build, [1] the
// injected-randomness one, each a list of kernel names ended by a null; an empty list means that build does not exist.
// Parts 1 and 2 are separate programs so that an env that never uses one family never pays its compile time.
enum { kPartRow = 0, kPartPlanes = 1, kPartRecord = 2, kParts = 3 };
struct JitPart {
  const char* kernels[2][3];
  bool two_sel_planes;   // not built for networks with a third selection plane (genes with more than 4 predictors)
};
static const JitPart kJitParts[kParts] = {
    // kPartRow: the row-format step (attractor table in shared memory / hash set, global table or r_wrong), pbn_rollout
    {{{"pbn_step_sliced", "pbn_step_sliced_gen", jit::kRolloutKernel}, {"pbn_step_sliced", "pbn_step_sliced_gen"}}, false},
    // kPartPlanes: the plane-resident step, 4 and 8 warps per tile
    {{{"pbn_step_planes_w4", "pbn_step_planes_w8"}, {"pbn_step_planes_w4", "pbn_step_planes_w8"}}, true},
    // kPartRecord: pbn_rollout_record
    {{{jit::kRecordKernel}, {}}, false},
};

static bool part_exists(const jit::GenNet& g, int part, int injected) {
  return kJitParts[part].kernels[injected][0] && !(kJitParts[part].two_sel_planes && jit::sel_bits(g) == 3);
}

// Compile (or fetch from the cubin cache) and load one program of the handle's network.
static int load_program(pbn_handle* h, int part, int injected) {
  pbn_handle::JitProgram& m = h->jit[part][injected];
  if (m.lib) return PBN_OK;
  std::vector<char> cubin;
  std::string err, key;
  if (jit::compile(h->gen, injected != 0, part, &cubin, &err) != 0) return fail(PBN_ERR_JIT, "%s", err.c_str());
  cudaLibrary_t lib = nullptr;
  const int rc = acquire_module(h, cubin, !injected, &lib, &key);
  if (rc != PBN_OK) return rc;
  const char* const* names = kJitParts[part].kernels[injected];
  for (int i = 0; i < 3 && names[i]; ++i) {
    const cudaError_t e = cudaLibraryGetKernel(&m.kernel[i].k, lib, names[i]);
    if (e != cudaSuccess) {
      release_module(key);
      return fail(PBN_ERR_CUDA, "cudaLibraryGetKernel(%s): %s", names[i], cudaGetErrorString(e));
    }
  }
  m.lib = lib;
  m.key = key;
  if (part == kPartRow) {
    h->sliced_threads = jit::sliced_threads(h->gen);
    h->sliced_min_blocks = jit::sliced_min_blocks(h->gen);
  }
  return PBN_OK;
}

// Blocks of `block` threads (or tiles of `block` envs) over n, at most per_sm of them per SM.
static int grid_for(const pbn_handle* h, int64_t n, int block, int per_sm) {
  int64_t g = (n + block - 1) / block;
  const int64_t cap = (int64_t)h->num_sms * per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

static SlicedSmemLayout sliced_smem_layout(const NetParams& n, int W, int scratch_words) {
  const uint32_t stage_state_bytes = 1024u * 8u * (uint32_t)W;
  const uint32_t stage_act_bytes = (1024u * (uint32_t)n.bins + 127u) & ~127u;
  SlicedSmemLayout L{};
  uint32_t o = 0;
  L.surv_off = o;
  o += 16u;  // (the survival table stays in global memory)
  o = (o + 15u) & ~15u;
  L.rew_off = o;
  o += 80u;
  const uint32_t abytes = (uint32_t)(n.n_attr + 1) * 4u + (uint32_t)n.n_attr_states * W * 16u + 32u;
  // (large attractors go through the hash set, the wrong-attractor reward term through the table scan: both live in
  //  the kernel's out-of-line membership path, selected by clearing this flag)
  L.attractors_in_smem = (n.n_attr > 0 && abytes <= 32u * 1024u && !(n.attr_simple == 0u && n.ahash_tags != nullptr) && n.r_wrong == 0.0f) ? 1u : 0u;
  if (L.attractors_in_smem) {
    L.acare_off = o;
    o += (uint32_t)n.n_attr_states * W * 8u;
    L.aval_off = o;
    o += (uint32_t)n.n_attr_states * W * 8u;
    L.aoffs_off = o;
    o += (uint32_t)(n.n_attr + 1) * 4u;
    o = (o + 15u) & ~15u;
  } else if (n.n_attr > 0 && n.attr_simple == 0u && n.ahash_tags != nullptr && n.awild_any == 0u && n.r_wrong == 0.0f &&
             (uint32_t)n.n_attr * ((uint32_t)W * 16u + 4u) <= 16u * 1024u) {
    L.singles_in_smem = 1u;
    L.acare_off = o;
    o += (uint32_t)n.n_attr * W * 16u;
    L.aval_off = o;
    L.aoffs_off = o;
    o += (uint32_t)n.n_attr * 4u;
    o = (o + 15u) & ~15u;
  }
  L.scratch_off = o;
  o += (uint32_t)scratch_words * 4u;  // one scratch per CTA (= per tile)
  o = (o + 127u) & ~127u;
  L.stage_state_off = o;
  o += stage_state_bytes;
  L.stage_act_off = o;
  o += stage_act_bytes;
  L.mbar_off = o;
  o += 16u;
  L.total = o;
  return L;
}

static bool aligned_to(const void* p, size_t a) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % a) == 0; }

static int launch_sliced(pbn_handle* h, StepParams& p, bool injected, cudaStream_t stream) {
  const pbn_step_args& a = p.a;
  if (!aligned_to(a.state, 16) || !aligned_to(a.final_state, 16) || !aligned_to(a.target_id, 16) ||
      !aligned_to(a.reward, 16) || !aligned_to(a.t, 8) || !aligned_to(a.actions, 16) ||
      !aligned_to(a.terminated, 4) || !aligned_to(a.truncated, 4))
    return fail(PBN_ERR_INVALID, "sliced kernel needs 16-byte aligned state/actions/target_id/reward, 8-byte t, 4-byte flags");
  int rc = load_program(h, kPartRow, injected);
  if (rc != PBN_OK) return rc;
  SlicedSmemLayout L = sliced_smem_layout(h->net, h->W, jit::scratch_words(h->gen));
  if (L.total > 227u * 1024u) return fail(PBN_ERR_UNSUPPORTED, "sliced kernel needs %u B of shared memory", L.total);
  pbn_handle::JitKernel& k = h->jit[kPartRow][injected].kernel[L.attractors_in_smem ? 0 : 1];
  if ((rc = ensure_dynamic_smem(reinterpret_cast<const void*>(k.k), L.total, &k.smem_opt_in)) != PBN_OK) return rc;
  // one CTA per 1024-env tile; beyond a few waves the CTAs loop over tiles
  void* args[] = {&p, &L};
  return launch(h, k.k, grid_for(h, a.n_envs, 1024, h->sliced_min_blocks * 8), h->sliced_threads, L.total, stream,
                a.flags & PBN_STEP_PDL, args);
}

// Which networks / attractor tables the plane-resident kernel takes (include/pbn_b200.h "Plane-resident env state").
static int resident_supported(const pbn_handle* h) {
  if (h->kernel != PBN_KERNEL_SLICED) return fail(PBN_ERR_UNSUPPORTED, "plane-resident state needs the sliced kernel");
  if (h->net.n_attr > 254) return fail(PBN_ERR_UNSUPPORTED, "plane-resident state: %d attractors > 254", h->net.n_attr);
  if (h->net.n_attr_states >= (1 << 24)) return fail(PBN_ERR_UNSUPPORTED, "plane-resident state: %d attractor table entries >= 2^24", h->net.n_attr_states);
  if (h->net.r_wrong != 0.0f) return fail(PBN_ERR_UNSUPPORTED, "plane-resident state: the wrong-attractor reward term (r_wrong) needs the row-format kernels");
  if (jit::sel_bits(h->gen) == 3) return fail(PBN_ERR_UNSUPPORTED, "plane-resident state: genes with more than 4 predictors need the row-format kernels");
  if (h->net.n_attr > 0 && !h->net.attr_simple && h->net.n_attr_states > 256)
    return fail(PBN_ERR_UNSUPPORTED, "plane-resident state: attractor table with %d (care, value) entries > 256 and several states per attractor", h->net.n_attr_states);
  return PBN_OK;
}

static int launch_planes(pbn_handle* h, StepParams& p, bool injected, cudaStream_t stream) {
  const pbn_step_args& a = p.a;
  int rc = resident_supported(h);
  if (rc != PBN_OK) return rc;
  if (!aligned_to(a.resident, 128) || !aligned_to(a.reward, 16) || !aligned_to(a.actions, 4) || !aligned_to(a.terminated, 4) || !aligned_to(a.truncated, 4))
    return fail(PBN_ERR_INVALID, "plane-resident step needs a 128-byte aligned block, 16-byte aligned reward, 4-byte aligned actions / flags");
  if ((rc = load_program(h, kPartPlanes, injected)) != PBN_OK) return rc;
  const NetParams& n = h->net;
  const int N = n.n_genes, NW = (N + 31) / 32;
  // 4 warps per tile (the selection planes stay in registers) for one-word states; 8 warps per tile where the
  // planes of a group would not fit the register file (N > 32: they are handed over through shared memory).  Both draw
  // the same streams.  (Measured with one shared code module per process, chained sequences: 3.69 vs 3.81 us per
  // 2^17-env step and 5.70 vs 6.51 us per 2^18-env step for 4 vs 8 warps.)
  int v = N > 32 ? 1 : 0;
  if (const char* env = getenv("PBN_B200_PLANES_WARPS")) v = atoi(env) == 8 ? 1 : 0;
  const int maxs4 = (jit::n_sel_slots(h->gen) + 3) / 4 > 0 ? (jit::n_sel_slots(h->gen) + 3) / 4 : 1;
  PlanesLayout L{};
  // dummy row | IN block | O planes | misc | reset job list | reset draws | SELX (8-warp variant)   (step_planes.cuh)
  uint32_t o = (uint32_t)(32 + 32 * resident_rows(N) + 32 * N + 256 + 512 + 1024 + (v ? 4 * maxs4 * 2 * 32 : 0)) * 4u;
  const uint32_t tab = (uint32_t)n.n_attr_states * NW * 4u * (n.attr_simple ? 1u : 2u) + (uint32_t)(n.n_attr + 1) * 4u + (uint32_t)n.n_attr_states + 64u;
  L.attr_in_smem = (n.n_attr > 0 && (tab <= 24u * 1024u || !n.attr_simple)) ? 1u : 0u;
  if (L.attr_in_smem) {
    L.aval_off = o;
    o += (uint32_t)n.n_attr_states * NW * 4u;
    L.acare_off = o;
    if (!n.attr_simple) o += (uint32_t)n.n_attr_states * NW * 4u;
    L.aoffs_off = o;
    o += (uint32_t)(n.n_attr + 1) * 4u;
    L.eattr_off = o;
    if (!n.attr_simple) o += (uint32_t)n.n_attr_states;
    o = (o + 15u) & ~15u;
  }
  L.total = o;
  if (L.total > 227u * 1024u) return fail(PBN_ERR_UNSUPPORTED, "plane-resident kernel needs %u B of shared memory", L.total);
  pbn_handle::JitKernel& k = h->jit[kPartPlanes][injected].kernel[v];
  if ((rc = ensure_dynamic_smem(reinterpret_cast<const void*>(k.k), L.total, &k.smem_opt_in)) != PBN_OK) return rc;
  // One tile per CTA.  (CTAs that walk two tiles were the better form for tile-chained sequences while every handle ran
  // its own copy of the kernel code -- 7.1 vs 7.6 us per 2^17-env step; with the shared module one tile per CTA wins,
  // 3.8 vs 4.25 us.)
  void* args[] = {&p, &L};
  return launch(h, k.k, grid_for(h, a.n_envs, 1024, 64), v ? 256u : 128u, L.total, stream, a.flags & PBN_STEP_PDL, args);
}

extern "C" {

const char* pbn_last_error(void) { return g_err; }
const char* pbn_version(void) { return "pbn_b200 0.1 (sm_100a)"; }

int pbn_kernel_kind(const pbn_handle* h) { return h ? h->kernel : PBN_ERR_INVALID; }
int pbn_words_per_state(const pbn_handle* h) { return h ? h->W : PBN_ERR_INVALID; }
int pbn_launch_count(const pbn_handle* h, uint64_t* out) {
  if (!h || !out) return fail(PBN_ERR_INVALID, "pbn_launch_count: null argument");
  *out = h->launches;
  return PBN_OK;
}

void pbn_destroy(pbn_handle* h) {
  if (!h) return;
  {
    DeviceGuard g(h->device);
    cudaFree(h->d_func_offset);
    cudaFree(h->d_funcs);
    cudaFree(h->d_func_cum);
    cudaFree(h->d_survival);
    cudaFree(h->d_attr_offset);
    cudaFree(h->d_attr_care);
    cudaFree(h->d_attr_val);
    cudaFree(h->d_pair_cum);
    cudaFree(h->d_ahash_tags);
    cudaFree(h->d_ahash_state);
    cudaFree(h->d_ahash_attr);
    cudaFree(h->d_awild_offset);
    cudaFree(h->d_awild_entry);
    cudaFree(h->d_ticket);
    cudaFree(h->d_surv_sliced);
    cudaFree(h->d_wide);
    cudaFree(h->d_wide_lut);
    for (auto& part : h->jit)
      for (auto& m : part) release_module(m.key);
    for (int c = 0; c < pbn_handle::kMaxLanes; ++c) {
      if (h->s_lane[c]) cudaStreamDestroy(h->s_lane[c]);
      if (h->ev_k[c]) cudaEventDestroy(h->ev_k[c]);
    }
    for (auto& g : h->host_graph)
      if (g.exec) cudaGraphExecDestroy(g.exec);
    if (h->s_origin) cudaStreamDestroy(h->s_origin);
    if (h->ev_done) cudaEventDestroy(h->ev_done);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_entry) cudaEventDestroy(h->ev_entry);
  }
  delete h;
}

int pbn_create(const pbn_net_desc* d, pbn_handle** out) {
  if (!d || !out) return fail(PBN_ERR_INVALID, "pbn_create: null argument");
  *out = nullptr;
  const int N = d->n_genes, F = d->n_funcs;
  if (N < 1 || N > PBN_MAX_GENES) return fail(PBN_ERR_INVALID, "n_genes=%d outside 1..%d", N, PBN_MAX_GENES);
  if (F < N || !d->func_offset || !d->func_arity || !d->func_inputs || !d->func_lut || !d->func_cum)
    return fail(PBN_ERR_INVALID, "function tables missing or n_funcs=%d < n_genes=%d", F, N);
  if (d->bins < 1 || d->bins > PBN_MAX_BINS) return fail(PBN_ERR_INVALID, "bins=%d outside 1..%d", d->bins, PBN_MAX_BINS);
  if (d->horizon < 0 || d->horizon > 65535) return fail(PBN_ERR_INVALID, "horizon=%d outside 0..65535", d->horizon);
  if (d->perturb_mode < PBN_PERT_NONE || d->perturb_mode > PBN_PERT_C)
    return fail(PBN_ERR_INVALID, "perturb_mode=%d unknown", d->perturb_mode);
  if (!(d->perturb_p >= 0.0f && d->perturb_p < 1.0f)) return fail(PBN_ERR_INVALID, "perturb_p=%g outside [0,1)", d->perturb_p);
  if (d->func_offset[0] != 0 || d->func_offset[N] != F) return fail(PBN_ERR_INVALID, "func_offset is not a CSR over n_funcs");
  if (N > 4 * 32) return fail(PBN_ERR_INVALID, "too many genes");

  std::vector<FuncDesc> funcs(F);
  std::vector<WideDesc> wides((size_t)(d->n_wide > 0 ? d->n_wide : 0));
  if (d->n_wide < 0 || (d->n_wide > 0 && (!d->wide_inputs || !d->wide_lut_offset || !d->wide_lut)))
    return fail(PBN_ERR_INVALID, "n_wide=%d but wide tables missing", d->n_wide);
  uint32_t sel_block_mask = 0, max_arity = 0;
  for (int i = 0; i < N; ++i) {
    const int f0 = d->func_offset[i], f1 = d->func_offset[i + 1];
    if (f1 <= f0 || f1 > F) return fail(PBN_ERR_INVALID, "gene %d has no predictor function", i);
    if (f1 - f0 > 1) sel_block_mask |= 1u << (i >> 2);
    for (int f = f0; f < f1; ++f) {
      const int k = d->func_arity[f];
      if (k > PBN_MAX_WIDE_ARITY) return fail(PBN_ERR_UNSUPPORTED, "function %d has arity %d > %d", f, k, PBN_MAX_WIDE_ARITY);
      max_arity = k > (int)max_arity ? (uint32_t)k : max_arity;
      if (k > PBN_MAX_ARITY) {  // wide predictor: multi-word truth table
        const uint64_t v = d->func_lut[f];
        if (v >= (uint64_t)d->n_wide) return fail(PBN_ERR_INVALID, "function %d: wide index %llu out of range", f, (unsigned long long)v);
        const int64_t words = (int64_t)d->wide_lut_offset[v + 1] - d->wide_lut_offset[v];
        if (d->wide_lut_offset[v] < 0 || words != (1ll << (k - 6))) return fail(PBN_ERR_INVALID, "function %d: wide truth table has %lld words, arity %d needs %lld", f, (long long)words, k, 1ll << (k - 6));
        WideDesc& wd = wides[v];
        memset(&wd, 0, sizeof(wd));
        for (int j = 0; j < k; ++j) {
          wd.in[j] = d->wide_inputs[v * 16 + j];
          if (wd.in[j] >= N) return fail(PBN_ERR_INVALID, "function %d input %d out of range", f, j);
        }
        wd.lut_off = (uint32_t)d->wide_lut_offset[v];
        wd.arity = (uint32_t)k;
        funcs[f].lut_lo = (uint32_t)v;
        funcs[f].lut_hi = 0;
        funcs[f].in03 = 0;
        funcs[f].in47 = kWideMarker;
        continue;
      }
      uint8_t in[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      for (int j = 0; j < k; ++j) {
        in[j] = d->func_inputs[f * PBN_FUNC_INPUT_STRIDE + j];
        if (in[j] >= N) return fail(PBN_ERR_INVALID, "function %d input %d out of range", f, j);
      }
      const uint64_t lut = d->func_lut[f];
      const uint64_t kmask = (1ull << k) - 1ull;
      uint64_t rep = 0;
      for (int a = 0; a < 64; ++a) rep |= ((lut >> (a & kmask)) & 1ull) << a;
      funcs[f].lut_lo = (uint32_t)rep;
      funcs[f].lut_hi = (uint32_t)(rep >> 32);
      funcs[f].in03 = in[0] | (in[1] << 8) | (in[2] << 16) | ((uint32_t)in[3] << 24);
      funcs[f].in47 = in[4] | (in[5] << 8) | (in[6] << 16) | ((uint32_t)in[7] << 24);
    }
  }
  std::vector<uint32_t> surv(N + 1);
  for (int j = 0; j <= N; ++j) {
    if (d->survival) {
      surv[j] = d->survival[j];
    } else {
      const double v = std::pow(1.0 - (double)d->perturb_p, (double)j) * 4294967296.0;
      surv[j] = v >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)v;
    }
  }

  std::string why;
  bool can_slice = jit::eligible(d, &why);
  int kernel = d->kernel;
  if (kernel == PBN_KERNEL_AUTO) kernel = can_slice ? PBN_KERNEL_SLICED : PBN_KERNEL_SCALAR;
  if (kernel != PBN_KERNEL_SCALAR && kernel != PBN_KERNEL_SLICED) return fail(PBN_ERR_INVALID, "kernel kind %d unknown", d->kernel);
  if (kernel == PBN_KERNEL_SLICED && !can_slice)
    return fail(PBN_ERR_UNSUPPORTED, "network not eligible for the sliced kernel: %s", why.c_str());

  int ndev = 0;
  PBN_CUDA(cudaGetDeviceCount(&ndev));
  if (d->device < 0 || d->device >= ndev) return fail(PBN_ERR_INVALID, "device %d not present (%d visible)", d->device, ndev);
  DeviceGuard guard(d->device);
  if (!guard.ok) return fail(PBN_ERR_CUDA, "cannot select device %d", d->device);

  pbn_handle* h = new (std::nothrow) pbn_handle();
  if (!h) return fail(PBN_ERR_INVALID, "out of host memory");
  h->device = d->device;
  h->W = N <= 64 ? 1 : 2;
  h->kernel = kernel;
  h->perturb_p = d->perturb_p;
  cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, d->device);

  int rc;
  if ((rc = upload(&h->d_func_offset, d->func_offset, (size_t)N + 1)) != PBN_OK ||
      (rc = upload(&h->d_funcs, funcs.data(), (size_t)F)) != PBN_OK ||
      (rc = upload(&h->d_func_cum, d->func_cum, (size_t)F)) != PBN_OK ||
      (rc = upload(&h->d_survival, surv.data(), (size_t)N + 1)) != PBN_OK) {
    pbn_destroy(h);
    return rc;
  }
  if (d->n_wide > 0) {
    if ((rc = upload(&h->d_wide, wides.data(), wides.size())) != PBN_OK ||
        (rc = upload(&h->d_wide_lut, d->wide_lut, (size_t)d->wide_lut_offset[d->n_wide])) != PBN_OK) {
      pbn_destroy(h);
      return rc;
    }
  }
  {
    const unsigned int zero = 0;
    if ((rc = upload(&h->d_ticket, &zero, 1)) != PBN_OK) {
      pbn_destroy(h);
      return rc;
    }
  }
  if (kernel == PBN_KERNEL_SLICED) {
    h->gen = jit::gen_net_from_desc(d);
    const std::vector<uint32_t> ss = jit::sliced_survival(d->perturb_p, N);
    h->surv_sliced_host = ss;
    if ((rc = upload(&h->d_surv_sliced, ss.data(), ss.size())) != PBN_OK || (rc = load_program(h, kPartRow, 0)) != PBN_OK) {
      pbn_destroy(h);
      return rc;
    }
  }
  NetParams& n = h->net;
  n.surv_sliced = h->d_surv_sliced;
  n.wide = h->d_wide;
  n.wide_lut = h->d_wide_lut;
  n.func_offset = h->d_func_offset;
  n.funcs = h->d_funcs;
  n.func_cum = h->d_func_cum;
  n.survival = h->d_survival;
  n.n_genes = N;
  n.n_funcs = F;
  n.bins = d->bins;
  n.horizon = d->horizon;
  n.pert_mode = d->perturb_mode;  // injected masks apply even when perturb_p == 0
  n.pert_rng = d->perturb_p > 0.0f ? 1u : 0u;
  n.pert_inv_log2 = d->perturb_p > 0.0 ? (float)(1.0 / std::log2(1.0 - d->perturb_p)) : 0.0f;
  n.r_success = d->r_success;
  n.r_wrong = d->r_wrong;
  n.r_step = d->r_step;
  n.r_action = d->r_action;
  n.k0 = (uint32_t)d->seed;
  n.k1 = (uint32_t)(d->seed >> 32);
  for (int r = 0; r < 10; ++r) {
    n.rk[2 * r] = n.k0 + (uint32_t)r * 0x9E3779B9u;
    n.rk[2 * r + 1] = n.k1 + (uint32_t)r * 0xBB67AE85u;
  }
  n.sel_block_mask = sel_block_mask;
  n.max_arity = max_arity;
  n.pair_last = 0;
  *out = h;
  return PBN_OK;
}

int pbn_update_attractors(pbn_handle* h, const int32_t* attr_offset, const uint64_t* care, const uint64_t* value,
                          int32_t n_attractors, const uint32_t* pair_cum, void* stream_) {
  if (!h) return fail(PBN_ERR_INVALID, "null handle");
  if (n_attractors < 0 || n_attractors > 46340) return fail(PBN_ERR_INVALID, "n_attractors=%d out of range", n_attractors);
  if (n_attractors > 0 && (!attr_offset || !care || !value)) return fail(PBN_ERR_INVALID, "attractor tables missing");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  const int A = n_attractors;
  const int S = A > 0 ? attr_offset[A] : 0;
  if (A > 0) {
    if (attr_offset[0] != 0) return fail(PBN_ERR_INVALID, "attr_offset[0] != 0");
    for (int a = 0; a < A; ++a)
      if (attr_offset[a + 1] <= attr_offset[a]) return fail(PBN_ERR_INVALID, "attractor %d is empty", a);
  }
  int rc;
  if ((rc = update_table(&h->d_attr_offset, &h->cap_attr_offset, attr_offset, (size_t)(A > 0 ? A + 1 : 0), stream)) != PBN_OK) return rc;
  if ((rc = update_table(&h->d_attr_care, &h->cap_attr_care, care, (size_t)S * h->W, stream)) != PBN_OK) return rc;
  if ((rc = update_table(&h->d_attr_val, &h->cap_attr_val, value, (size_t)S * h->W, stream)) != PBN_OK) return rc;
  int pair_last = 0;
  if (pair_cum && A > 0) {
    uint32_t prev = 0;
    for (int k = 0; k < A * A; ++k) {
      if (pair_cum[k] < prev) return fail(PBN_ERR_INVALID, "pair_cum is not non-decreasing at %d", k);
      if (pair_cum[k] > prev || (k == 0 && pair_cum[0] > 0)) pair_last = k;
      prev = pair_cum[k];
    }
    if ((rc = update_table(&h->d_pair_cum, &h->cap_pair_cum, pair_cum, (size_t)A * A, stream)) != PBN_OK) return rc;
  }
  NetParams& n = h->net;
  n.attr_offset = h->d_attr_offset;
  n.attr_care = h->d_attr_care;
  n.attr_val = h->d_attr_val;
  n.pair_cum = (pair_cum && A > 0) ? h->d_pair_cum : nullptr;
  n.n_attr = A;
  n.n_attr_states = S;
  n.pair_last = pair_last;
  bool simple = A > 0 && S == A;
  for (int e = 0; simple && e < S; ++e)
    for (int w = 0; w < h->W; ++w) {
      const int nbits = n.n_genes - 64 * w;
      const uint64_t full = nbits >= 64 ? ~0ull : ((1ull << nbits) - 1ull);
      if (care[(size_t)e * h->W + w] != full) simple = false;
    }
  n.attr_simple = simple ? 1u : 0u;

  // Hash set for tables with large attractors (an attractor of more than kHashMinStates = 64 states): membership becomes
  // one probe sequence instead of a scan over the attractor (pbn70 has an 8192-state attractor; model_tester.py:602-616).
  constexpr int kHashMinStates = 64;   // below that the scan over the attractor in shared memory is the faster test
  int largest = 0;
  for (int a = 0; a < A; ++a) largest = std::max(largest, attr_offset[a + 1] - attr_offset[a]);
  n.ahash_tags = nullptr;
  n.ahash_state = nullptr;
  n.ahash_attr = nullptr;
  n.awild_offset = nullptr;
  n.awild_entry = nullptr;
  n.ahash_mask = 0;
  n.awild_any = 0;
  if (!simple && largest > kHashMinStates) {
    const int W = h->W;
    std::vector<int32_t> wild_off(A + 1, 0), wild_entry;
    std::vector<int> exact;   // entry indices
    for (int a = 0; a < A; ++a) {
      for (int e = attr_offset[a]; e < attr_offset[a + 1]; ++e) {
        bool full = true;
        for (int w = 0; w < W; ++w) {
          const int nbits = n.n_genes - 64 * w;
          const uint64_t m = nbits >= 64 ? ~0ull : ((1ull << nbits) - 1ull);
          if (care[(size_t)e * W + w] != m) full = false;
        }
        if (full) exact.push_back(e); else wild_entry.push_back(e);
      }
      wild_off[a + 1] = (int32_t)wild_entry.size();
    }
    size_t cap = 64;
    // at most 1/16 full (1/4 beyond 4 M slots): the step kernels decide a membership test inline when the first
    // probe finds an empty slot, and every occupied one sends the whole warp through the out-of-line probe loop
    while (cap < 4 * exact.size() + 2 || (cap < 16 * exact.size() + 2 && cap < (1u << 22))) cap *= 2;
    std::vector<unsigned long long> tags(cap, 0ull);
    std::vector<uint64_t> states(cap * W, 0ull);
    std::vector<int32_t> owner(cap, -1);
    std::vector<int32_t> attr_of(S);
    for (int a = 0; a < A; ++a)
      for (int e = attr_offset[a]; e < attr_offset[a + 1]; ++e) attr_of[e] = a;
    for (int e : exact) {
      const uint64_t* st = value + (size_t)e * W;
      const uint64_t tag = attr_tag(st, W);
      size_t slot = attr_slot(tag, (uint32_t)(cap - 1));
      while (tags[slot] != 0ull) slot = (slot + 1) & (cap - 1);
      tags[slot] = tag;
      for (int w = 0; w < W; ++w) states[slot * W + w] = st[w];
      owner[slot] = attr_of[e];
    }
    if (wild_entry.empty()) wild_entry.push_back(0);   // never an empty upload
    if ((rc = update_table(&h->d_ahash_tags, &h->cap_ahash_tags, tags.data(), tags.size(), stream)) != PBN_OK ||
        (rc = update_table(&h->d_ahash_state, &h->cap_ahash_state, states.data(), states.size(), stream)) != PBN_OK ||
        (rc = update_table(&h->d_ahash_attr, &h->cap_ahash_attr, owner.data(), owner.size(), stream)) != PBN_OK ||
        (rc = update_table(&h->d_awild_offset, &h->cap_awild_offset, wild_off.data(), wild_off.size(), stream)) != PBN_OK ||
        (rc = update_table(&h->d_awild_entry, &h->cap_awild_entry, wild_entry.data(), wild_entry.size(), stream)) != PBN_OK)
      return rc;
    // (pageable sources: cudaMemcpyAsync has staged them before it returned, the local vectors may go)
    n.ahash_tags = h->d_ahash_tags;
    n.ahash_state = h->d_ahash_state;
    n.ahash_attr = h->d_ahash_attr;
    n.awild_offset = h->d_awild_offset;
    n.awild_entry = h->d_awild_entry;
    n.ahash_mask = (uint32_t)(cap - 1);
    n.awild_any = wild_off[A] > 0 ? 1u : 0u;
  }
  return PBN_OK;
}

int pbn_attractor_hash_slots(const pbn_handle* h) { return h ? (h->net.ahash_tags ? (int)h->net.ahash_mask + 1 : 0) : PBN_ERR_INVALID; }

static int step_common(pbn_handle* h, const pbn_step_args* a, void* stream_, bool injected) {
  if (!h || !a) return fail(PBN_ERR_INVALID, "null argument");
  if (a->n_envs < 0) return fail(PBN_ERR_INVALID, "n_envs=%lld", (long long)a->n_envs);
  if (a->n_envs == 0) return PBN_OK;
  if (a->resident) {
    if (a->state || a->target_id || a->t || a->final_state)
      return fail(PBN_ERR_INVALID, "plane-resident step: state / target_id / t / final_state must be null (the block holds them)");
    if (h->kernel != PBN_KERNEL_SLICED) return fail(PBN_ERR_UNSUPPORTED, "plane-resident state needs the sliced kernel");
  } else if (!a->state) {
    return fail(PBN_ERR_INVALID, "state is null");
  }
  if (injected && !a->sel) return fail(PBN_ERR_INVALID, "pbn_step_injected needs args->sel");
  if (!injected && (a->sel || a->pert_mask)) return fail(PBN_ERR_INVALID, "pbn_step: sel/pert_mask must be null (use pbn_step_injected)");
  if (a->env_offset < 0 || (a->env_offset & 1023)) return fail(PBN_ERR_INVALID, "env_offset=%lld must be a non-negative multiple of 1024", (long long)a->env_offset);
  if (a->target_id && h->net.n_attr == 0) return fail(PBN_ERR_NO_ATTRACTORS, "target_id given but no attractor table uploaded");
  {
    const uint32_t known = PBN_STEP_AUTORESET | PBN_STEP_PDL | PBN_STEP_NO_COUNT | PBN_STEP_CHAIN | (jit::profile_build() ? 0x80000000u : 0u);
    if (a->flags & ~known) return fail(PBN_ERR_INVALID, "unknown flag bits 0x%x", a->flags & ~known);
  }
  if ((a->flags & PBN_STEP_PDL) && !a->step_ctr_dev) return fail(PBN_ERR_INVALID, "PBN_STEP_PDL needs step_ctr_dev");
  if ((a->flags & PBN_STEP_CHAIN) && (!a->resident || !(a->flags & PBN_STEP_PDL) || injected))
    return fail(PBN_ERR_INVALID, "PBN_STEP_CHAIN needs args->resident and PBN_STEP_PDL (own-RNG steps)");
  if (a->flags & PBN_STEP_AUTORESET) {
    if (h->net.n_attr == 0) return fail(PBN_ERR_NO_ATTRACTORS, "auto-reset needs pbn_update_attractors first");
    if (!a->resident && (!a->target_id || !a->t)) return fail(PBN_ERR_INVALID, "auto-reset needs target_id and t");
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  StepParams p;
  p.a = *a;
  p.n = h->net;
  p.ticket = h->d_ticket;
  if (h->kernel == PBN_KERNEL_SLICED)
    return a->resident ? launch_planes(h, p, injected, stream) : launch_sliced(h, p, injected, stream);
  const ScalarSmemLayout L = scalar_smem_layout(h->net, h->W);
  if (L.total > 200u * 1024u) return fail(PBN_ERR_UNSUPPORTED, "network tables need %u B of shared memory", L.total);
  // [W - 1][predictor arity: up to 4, up to 6, wider]
  static const decltype(&step_scalar_kernel<1, 4>) scalar_kernel[2][3] = {
      {step_scalar_kernel<1, 4>, step_scalar_kernel<1, 6>, step_scalar_kernel<1, 16>},
      {step_scalar_kernel<2, 4>, step_scalar_kernel<2, 6>, step_scalar_kernel<2, 16>}};
  const auto k = scalar_kernel[h->W - 1][h->net.max_arity > PBN_MAX_ARITY ? 2 : h->net.max_arity > 4 ? 1 : 0];
  const int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(k), L.total, &h->scalar_smem_opt_in);
  if (rc != PBN_OK) return rc;
  return launch(h, k, grid_for(h, a->n_envs, 256, 8), 256, L.total, stream, false, p, L);
}

int64_t pbn_jit_source(const pbn_net_desc* d, int injected, char* buf, int64_t len) {
  if (!d || d->n_genes < 1 || !d->func_offset) return fail(PBN_ERR_INVALID, "bad descriptor");
  std::string why;
  if (!jit::eligible(d, &why)) return fail(PBN_ERR_UNSUPPORTED, "not eligible for the sliced kernel: %s", why.c_str());
  std::string gen_h, upd;
  jit::generate(jit::gen_net_from_desc(d), injected != 0, &gen_h, &upd);
  const std::string all = "// ---- net_gen.cuh\n" + gen_h + "// ---- net_update.inc\n" + upd;
  if (buf && len > 0) {
    const size_t n = all.size() < (size_t)(len - 1) ? all.size() : (size_t)(len - 1);
    memcpy(buf, all.data(), n);
    buf[n] = 0;
  }
  return (int64_t)all.size();
}

int pbn_jit_precompile(const pbn_net_desc* d) {
  if (!d || d->n_genes < 1 || !d->func_offset) return fail(PBN_ERR_INVALID, "bad descriptor");
  std::string why;
  if (!jit::eligible(d, &why)) return fail(PBN_ERR_UNSUPPORTED, "not eligible for the sliced kernel: %s", why.c_str());
  const jit::GenNet g = jit::gen_net_from_desc(d);
  for (int inj = 0; inj < 2; ++inj) {
    std::vector<char> cubin;
    std::string err;
    for (int part = 0; part < kParts; ++part)
      if (part_exists(g, part, inj) && jit::compile(g, inj != 0, part, &cubin, &err) != 0) return fail(PBN_ERR_JIT, "%s", err.c_str());
  }
  return PBN_OK;
}

int pbn_step(pbn_handle* h, const pbn_step_args* a, void* stream) { return step_common(h, a, stream, false); }

// Checks the projection of a recording call and copies it into proj[12].
static int record_projection(const pbn_handle* h, const char* who, const int32_t* proj_genes, int32_t n_proj, int32_t* proj) {
  if (n_proj < 0 || n_proj > 12) return fail(PBN_ERR_INVALID, "%s: n_proj = %d, must be in [0, 12]", who, n_proj);
  if (n_proj > 0 && !proj_genes) return fail(PBN_ERR_INVALID, "%s: proj_genes is NULL", who);
  for (int j = 0; j < 12; ++j) proj[j] = 0;
  for (int j = 0; j < n_proj; ++j) {
    const int32_t g = proj_genes[j];
    if (g < 0 || g >= h->net.n_genes) return fail(PBN_ERR_INVALID, "%s: projection gene %d outside [0, %d)", who, g, h->net.n_genes);
    for (int i = 0; i < j; ++i)
      if (proj[i] == g) return fail(PBN_ERR_INVALID, "%s: projection gene %d appears twice", who, g);
    proj[j] = g;
  }
  return PBN_OK;
}

// pbn_rollout (rec = false: the rollout kernel of program kPartRow) and pbn_rollout_record (rec = true: program
// kPartRecord, which also takes the recording arguments).
static int rollout(pbn_handle* h, bool rec, uint64_t* state, int64_t n_steps, uint64_t step_ctr, int64_t env_offset,
                   int64_t n_envs, int32_t stride, const int32_t* proj_genes, int32_t n_proj, unsigned long long* gene_on,
                   unsigned long long* hist, unsigned long long* stats, void* stream_) {
  const char* who = rec ? "pbn_rollout_record" : "pbn_rollout";
  if (!h || !state) return fail(PBN_ERR_INVALID, "null argument");
  if (h->kernel != PBN_KERNEL_SLICED)
    return fail(PBN_ERR_UNSUPPORTED, "%s: the handle runs the scalar kernel (loop over %s)", who, rec ? "pbn_step + pbn_record_states" : "pbn_step");
  if (n_envs < 0 || n_steps < 0 || n_steps > 0x7FFFFFFF || env_offset < 0 || (env_offset & 1023)) return fail(PBN_ERR_INVALID, "bad n_envs / n_steps / env_offset");
  RecordParams q;
  if (rec) {
    if (stride < 1) return fail(PBN_ERR_INVALID, "%s: stride = %d, must be >= 1", who, stride);
    const int rc = record_projection(h, who, proj_genes, n_proj, q.proj);
    if (rc != PBN_OK) return rc;
  }
  if (n_envs == 0 || n_steps == 0) return PBN_OK;
  DeviceGuard guard(h->device);
  int rc = load_program(h, kPartRow, 0);
  if (rc == PBN_OK && rec) rc = load_program(h, kPartRecord, 0);
  if (rc != PBN_OK) return rc;
  const int N = h->net.n_genes, NW = (N + 31) / 32, NSEL = jit::n_sel_slots(h->gen);
  // the rollout's scratch, then the 2^n_proj histogram bins of the recording form
  const uint32_t smem = (uint32_t)(2 * NW * 1024 + jit::sel_bits(h->gen) * NSEL * 32 + 128 * (8 * N < 255 ? 1 : 2) + 32 + 8 + (rec ? 1 << n_proj : 0)) * 4u;
  if (smem > 227u * 1024u) return fail(PBN_ERR_UNSUPPORTED, "%s needs %u B of shared memory", who, smem);
  pbn_handle::JitKernel& k = rec ? h->jit[kPartRecord][0].kernel[0] : h->jit[kPartRow][0].kernel[2];
  if ((rc = ensure_dynamic_smem(reinterpret_cast<const void*>(k.k), smem, &k.smem_opt_in)) != PBN_OK) return rc;
  q.r.n = h->net;
  q.r.state = state;
  q.r.stats = stats;
  q.r.step_ctr = step_ctr;
  q.r.env_offset = env_offset;
  q.r.n_envs = n_envs;
  q.r.n_steps = (int32_t)n_steps;
  q.gene_on = gene_on;
  q.hist = hist;
  q.stride = stride;
  q.n_proj = n_proj;
  void* args[] = {rec ? static_cast<void*>(&q) : static_cast<void*>(&q.r)};
  return launch(h, k.k, grid_for(h, n_envs, 1024, h->sliced_min_blocks * 8), h->sliced_threads, smem,
                static_cast<cudaStream_t>(stream_), false, args);
}

int pbn_rollout(pbn_handle* h, uint64_t* state, int64_t n_steps, uint64_t step_ctr, int64_t env_offset, int64_t n_envs,
                unsigned long long* stats, void* stream) {
  return rollout(h, false, state, n_steps, step_ctr, env_offset, n_envs, 1, nullptr, 0, nullptr, nullptr, stats, stream);
}

int pbn_rollout_record(pbn_handle* h, uint64_t* state, int64_t n_steps, uint64_t step_ctr, int64_t env_offset,
                       int64_t n_envs, int32_t stride, const int32_t* proj_genes, int32_t n_proj,
                       unsigned long long* gene_on, unsigned long long* hist, unsigned long long* stats, void* stream) {
  return rollout(h, true, state, n_steps, step_ctr, env_offset, n_envs, stride, proj_genes, n_proj, gene_on, hist, stats,
                 stream);
}

int pbn_record_states(pbn_handle* h, const uint64_t* state, int64_t n_envs, const int32_t* proj_genes, int32_t n_proj,
                      unsigned long long* gene_on, unsigned long long* hist, void* stream_) {
  if (!h) return fail(PBN_ERR_INVALID, "null argument");
  if (n_envs < 0) return fail(PBN_ERR_INVALID, "pbn_record_states: n_envs < 0");
  if (n_envs > 0 && !state) return fail(PBN_ERR_INVALID, "pbn_record_states: state is NULL");
  RecordStatesParams q;
  int rc = record_projection(h, "pbn_record_states", proj_genes, n_proj, q.proj);
  if (rc != PBN_OK) return rc;
  if (n_envs == 0 || (!gene_on && !hist)) return PBN_OK;
  DeviceGuard guard(h->device);
  q.state = state;
  q.gene_on = gene_on;
  q.hist = hist;
  q.n_envs = n_envs;
  q.n_genes = h->net.n_genes;
  q.W = h->W;
  q.n_proj = n_proj;
  const uint32_t smem = (uint32_t)((hist ? (1u << n_proj) : 0u) * 4u + 128u * 8u);
  return launch(h, record_states_kernel, grid_for(h, n_envs, kRecordThreads, 4), kRecordThreads, smem,
                static_cast<cudaStream_t>(stream_), false, q);
}

// The step arguments of envs [e0, e0 + n) of a row-format batch; actions: the device actions of the whole batch or null.
static pbn_step_args env_range(const pbn_handle* h, const pbn_step_args* a, const uint8_t* actions, int64_t e0, int64_t n) {
  pbn_step_args s = *a;
  s.state = a->state + e0 * h->W;
  s.actions = actions ? actions + e0 * h->net.bins : nullptr;
  if (a->target_id) s.target_id = a->target_id + e0;
  if (a->source_id) s.source_id = a->source_id + e0;
  if (a->t) s.t = a->t + e0;
  if (a->reward) s.reward = a->reward + e0;
  if (a->terminated) s.terminated = a->terminated + e0;
  if (a->truncated) s.truncated = a->truncated + e0;
  if (a->final_state) s.final_state = a->final_state + e0 * h->W;
  s.env_offset = a->env_offset + e0;
  s.n_envs = n;
  return s;
}

// The device alias of a page-locked host buffer; null for a null or pageable one (the failed query's error is cleared).
static void* mapped(void* host) {
  void* dev = nullptr;
  if (host && (cudaHostGetDevicePointer(&dev, host, 0) != cudaSuccess || !dev)) {
    cudaGetLastError();
    dev = nullptr;
  }
  return dev;
}

// Envs [e0, e0 + n) of the export of a whole batch of W-word states.
static ExportArgs export_range(ExportArgs x, int W, int64_t e0, int64_t n) {
  const int64_t row[4] = {8 * W, 4, 1, 1};   // bytes per env of the state words, reward, terminated, truncated
  for (int k = 0; k < 4; ++k) {
    if (x.dst[k]) x.src[k] += e0 * row[k], x.dst[k] += e0 * row[k];
    x.bytes[k] = (unsigned long long)(n * row[k]);
  }
  x.state64 += e0 * W;
  if (x.state32) x.state32 += e0;
  if (x.term) x.term += e0;
  if (x.trunc) x.trunc += e0;
  if (x.done) x.done += e0;
  if (x.packed) x.packed += e0;
  x.n_envs = n;
  return x;
}

// Runs `enqueue` (one step's work, forked from and joined into h->s_origin) through the handle's graph cache, keyed by
// the (args, io) pair: the first call with a pair runs eagerly, the second (every kernel it needs is loaded by then)
// captures the work, and from the third on it is replayed as one graph launch.  The least recently used slot is evicted.
static int run_host_graph(pbn_handle* h, const pbn_step_args* a, const pbn_host_io* io, const std::function<int()>& enqueue) {
  pbn_handle::HostGraph* slot = nullptr;
  pbn_handle::HostGraph* lru = &h->host_graph[0];
  for (auto& g : h->host_graph) {
    if (g.seen && memcmp(&g.a, a, sizeof(*a)) == 0 && memcmp(&g.io, io, sizeof(*io)) == 0) slot = &g;
    if (g.last_use < lru->last_use) lru = &g;
  }
  if (!slot) {
    slot = lru;
    if (slot->exec) cudaGraphExecDestroy(slot->exec);
    *slot = pbn_handle::HostGraph{};
    memcpy(&slot->a, a, sizeof(*a));
    memcpy(&slot->io, io, sizeof(*io));
  }
  slot->last_use = ++h->host_graph_clock;
  if (slot->exec) {
    PBN_CUDA(cudaGraphLaunch(slot->exec, h->s_origin));
    h->launches += slot->launches;
  } else if (slot->seen >= 1) {
    const uint64_t launches_before = h->launches;
    cudaGraph_t graph = nullptr;
    PBN_CUDA(cudaStreamBeginCapture(h->s_origin, cudaStreamCaptureModeThreadLocal));
    const int rc = enqueue();
    const cudaError_t ce = cudaStreamEndCapture(h->s_origin, &graph);
    if (rc != PBN_OK) {
      if (graph) cudaGraphDestroy(graph);
      return rc;
    }
    if (ce != cudaSuccess) return fail(PBN_ERR_CUDA, "pbn_step_host: graph capture failed: %s", cudaGetErrorString(ce));
    const cudaError_t ie = cudaGraphInstantiate(&slot->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess) {
      slot->exec = nullptr;
      return fail(PBN_ERR_CUDA, "pbn_step_host: graph instantiation failed: %s", cudaGetErrorString(ie));
    }
    slot->launches = h->launches - launches_before;
    PBN_CUDA(cudaGraphLaunch(slot->exec, h->s_origin));
  } else {
    const int rc = enqueue();
    if (rc != PBN_OK) return rc;
  }
  slot->seen += 1;
  return PBN_OK;
}

int pbn_step_host(pbn_handle* h, const pbn_step_args* a, const pbn_host_io* io, void* stream_) {
  if (!h || !a || !io) return fail(PBN_ERR_INVALID, "null argument");
  if (a->n_envs < 0) return fail(PBN_ERR_INVALID, "n_envs=%lld", (long long)a->n_envs);
  if (a->n_envs == 0) return PBN_OK;
  if ((io->actions || io->actions16) && !io->actions_dev) return fail(PBN_ERR_INVALID, "pbn_step_host: actions given without actions_dev staging buffer");
  if (io->actions16 && (io->actions || !io->actions16_dev || h->net.bins != 3 || h->net.n_genes > 30))
    return fail(PBN_ERR_INVALID, "pbn_step_host: actions16 needs actions16_dev, no `actions`, bins == 3 and N <= 30");
  if (a->resident) return fail(PBN_ERR_UNSUPPORTED, "pbn_step_host works on the row-format arrays (export the resident block first)");
  if ((io->reward && !a->reward) || (io->terminated && !a->terminated) || (io->truncated && !a->truncated) || !a->state)
    return fail(PBN_ERR_INVALID, "pbn_step_host: a host output is requested whose device array is null");
  if (a->sel || a->pert_mask) return fail(PBN_ERR_INVALID, "pbn_step_host: sel/pert_mask must be null");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  // Results in page-locked host memory are written by the export kernel straight over PCIe, through the buffers' device
  // aliases (one launch per lane); pageable full-width results go through the copy engine (one cudaMemcpyAsync per
  // array and lane).  (Measured: letting the step kernel write the packed word straight into the mapped host buffer --
  // 1024 CTAs posting 16-byte writes -- is slower over PCIe, 0.200 ms per 2^20 envs, than the 16-CTA export kernel,
  // 0.176 ms.)
  const int W = h->W, bins = h->net.bins;
  ExportArgs all{};
  bool zero_copy = true;   // every requested full-width output is page-locked
  {
    void* const host[4] = {io->state, io->reward, io->terminated, io->truncated};
    const void* const dev[4] = {a->state, a->reward, a->terminated, a->truncated};
    for (int k = 0; k < 4; ++k) {
      all.src[k] = static_cast<const uint8_t*>(dev[k]);
      all.dst[k] = static_cast<uint8_t*>(mapped(host[k]));
      if (host[k] && !all.dst[k]) zero_copy = false;
    }
  }
  all.state64 = a->state;
  all.term = a->terminated;
  all.trunc = a->truncated;
  if (io->packed) {
    if (h->net.n_genes > 30 || !a->terminated || !a->truncated) return fail(PBN_ERR_INVALID, "pbn_step_host: packed needs N <= 30 and the terminated / truncated device arrays");
    if (!zero_copy || !(all.packed = static_cast<uint32_t*>(mapped(io->packed))))
      return fail(PBN_ERR_INVALID, "pbn_step_host: packed needs page-locked host memory for every output");
  }
  if (io->state32 || io->done) {
    if (io->state32 && h->net.n_genes > 32) return fail(PBN_ERR_INVALID, "pbn_step_host: state32 needs a network with N <= 32 (N=%d)", h->net.n_genes);
    if (io->done && (!a->terminated || !a->truncated)) return fail(PBN_ERR_INVALID, "pbn_step_host: done needs the terminated and truncated device arrays");
    all.state32 = static_cast<uint32_t*>(mapped(io->state32));
    all.done = static_cast<uint8_t*>(mapped(io->done));
    if (!zero_copy || (io->state32 && !all.state32) || (io->done && !all.done))
      return fail(PBN_ERR_INVALID, "pbn_step_host: state32/done need page-locked host memory for every output");
  }
  // Graph replay needs arguments that are the same from call to call -- a device step counter keeps the host part of
  // the counter constant -- and only mapped outputs: a pageable copy cannot be captured.
  const bool graphable = io->packed && io->actions16 && a->step_ctr_dev && !io->state && !io->reward && !io->terminated &&
                         !io->truncated && !io->state32 && !io->done;
  // Lanes: slices of whole tiles, each running upload -> step -> results in order on its own library stream, so nothing
  // inside a lane needs an event and PCIe (full duplex) carries one lane's upload under another lane's results.  Envs are
  // independent: the results do not depend on the number of lanes.  Measured on B200 / PCIe Gen5, packed form, 2^20
  // envs: replayed graph 0.166 / 0.158 / 0.161 / 0.148 / 0.158 ms with 1 / 2 / 3 / 4 / 6 lanes; stream launches
  // 0.175 / 0.169 / 0.167 / 0.173 / 0.189 ms.
  const int64_t E = a->n_envs, tiles = (E + 1023) / 1024;
  int64_t lanes = io->n_chunks > 0 ? io->n_chunks : (E < (1 << 18) ? 1 : (graphable ? 4 : 2));
  lanes = std::min<int64_t>(std::min<int64_t>(lanes, pbn_handle::kMaxLanes), tiles);
  const int64_t per = ((tiles + lanes - 1) / lanes) * 1024;
  // The lanes' step kernels run concurrently, so they cannot each advance a device step counter: they share one counter
  // value (PBN_STEP_NO_COUNT), and a counter the steps would advance themselves gets one launch that adds 1 after the join.
  const bool own_count = a->step_ctr_dev && !(a->flags & (PBN_STEP_PDL | PBN_STEP_NO_COUNT));
  if (!h->s_origin) PBN_CUDA(cudaStreamCreateWithFlags(&h->s_origin, cudaStreamNonBlocking));
  for (cudaEvent_t* ev : {&h->ev_entry, &h->ev_fork, &h->ev_done})
    if (!*ev) PBN_CUDA(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
  for (int c = 0; c < lanes; ++c) {
    if (!h->s_lane[c]) PBN_CUDA(cudaStreamCreateWithFlags(&h->s_lane[c], cudaStreamNonBlocking));
    if (!h->ev_k[c]) PBN_CUDA(cudaEventCreateWithFlags(&h->ev_k[c], cudaEventDisableTiming));
  }
  const uint8_t* actions = (io->actions || io->actions16) ? io->actions_dev : nullptr;
  auto enqueue = [&]() -> int {
    PBN_CUDA(cudaEventRecord(h->ev_fork, h->s_origin));
    for (int c = 0; c < lanes; ++c) {
      const int64_t e0 = c * per, n = std::min(per, E - e0);
      if (n <= 0) break;
      cudaStream_t S = h->s_lane[c];
      PBN_CUDA(cudaStreamWaitEvent(S, h->ev_fork, 0));
      if (io->actions) {
        PBN_CUDA(cudaMemcpyAsync(io->actions_dev + e0 * bins, io->actions + e0 * bins, (size_t)n * bins, cudaMemcpyHostToDevice, S));
      } else if (io->actions16) {
        PBN_CUDA(cudaMemcpyAsync(io->actions16_dev + e0, io->actions16 + e0, (size_t)n * 2, cudaMemcpyHostToDevice, S));
        const int rc = launch(h, unpack_actions16_kernel, grid_for(h, n / 4 + 1, 256, 4), 256, 0, S, false,
                              io->actions16_dev + e0, io->actions_dev + e0 * bins, n);
        if (rc != PBN_OK) return rc;
      }
      // PDL only orders kernels, which the lane's stream already does
      pbn_step_args s = env_range(h, a, actions, e0, n);
      s.flags = (a->flags & ~PBN_STEP_PDL) | PBN_STEP_NO_COUNT;
      int rc = step_common(h, &s, S, false);
      if (rc != PBN_OK) return rc;
      if (zero_copy) {
        if ((rc = launch(h, export_kernel, 16, 256, 0, S, false, export_range(all, W, e0, n))) != PBN_OK) return rc;
      } else {
        if (io->state) PBN_CUDA(cudaMemcpyAsync(io->state + e0 * W, a->state + e0 * W, (size_t)n * W * 8, cudaMemcpyDeviceToHost, S));
        if (io->reward) PBN_CUDA(cudaMemcpyAsync(io->reward + e0, a->reward + e0, (size_t)n * 4, cudaMemcpyDeviceToHost, S));
        if (io->terminated) PBN_CUDA(cudaMemcpyAsync(io->terminated + e0, a->terminated + e0, (size_t)n, cudaMemcpyDeviceToHost, S));
        if (io->truncated) PBN_CUDA(cudaMemcpyAsync(io->truncated + e0, a->truncated + e0, (size_t)n, cudaMemcpyDeviceToHost, S));
      }
      PBN_CUDA(cudaEventRecord(h->ev_k[c], S));
      PBN_CUDA(cudaStreamWaitEvent(h->s_origin, h->ev_k[c], 0));
    }
    return own_count ? launch(h, advance_counter_kernel, 1, 1, 0, h->s_origin, false, a->step_ctr_dev, 1ull) : PBN_OK;
  };
  // the staging buffers and device arrays may still be in use by earlier work on the caller's stream
  PBN_CUDA(cudaEventRecord(h->ev_entry, stream));
  PBN_CUDA(cudaStreamWaitEvent(h->s_origin, h->ev_entry, 0));
  const int rc = graphable ? run_host_graph(h, a, io, enqueue) : enqueue();
  if (rc != PBN_OK) return rc;
  g_last_advance = own_count ? h : nullptr;
  PBN_CUDA(cudaEventRecord(h->ev_done, h->s_origin));
  PBN_CUDA(cudaStreamWaitEvent(stream, h->ev_done, 0));   // later work on the caller's stream sees the step
  PBN_CUDA(cudaEventSynchronize(h->ev_done));
  return PBN_OK;
}
int pbn_step_injected(pbn_handle* h, const pbn_step_args* a, void* stream) { return step_common(h, a, stream, true); }

int pbn_reward_table(const pbn_handle* h, float* out, int32_t n) {
  if (!h || !out) return fail(PBN_ERR_INVALID, "null argument");
  const int bins = h->net.bins;
  if (n < 2 * (bins + 1)) return fail(PBN_ERR_INVALID, "reward table has %d entries, buffer holds %d", 2 * (bins + 1), n);
  if (h->net.r_wrong != 0.0f) return fail(PBN_ERR_UNSUPPORTED, "with r_wrong != 0 the reward is not a function of (flips, terminated)");
  for (int hit = 0; hit < 2; ++hit)
    for (int nf = 0; nf <= bins; ++nf) {
      volatile float base = h->net.r_action * (float)nf;   // two separately rounded fp32 operations, as on the device
      base = h->net.r_step + base;
      out[nf + (bins + 1) * hit] = hit ? (float)(base + h->net.r_success) : base;
    }
  return PBN_OK;
}

int pbn_reset(pbn_handle* h, uint64_t* state, int32_t* target_id, int32_t* source_id, uint16_t* t,
              const uint8_t* done_mask, uint64_t step_ctr, int64_t env_offset, int64_t n_envs, void* stream_) {
  if (!h) return fail(PBN_ERR_INVALID, "null handle");
  if (n_envs < 0 || !state) return fail(PBN_ERR_INVALID, "bad arguments");
  if (n_envs == 0) return PBN_OK;
  if (h->net.n_attr == 0) return fail(PBN_ERR_NO_ATTRACTORS, "pbn_reset needs pbn_update_attractors first");
  if (env_offset < 0 || (env_offset & 1023)) return fail(PBN_ERR_INVALID, "env_offset must be a non-negative multiple of 1024");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, h->W == 1 ? reset_kernel<1> : reset_kernel<2>, grid_for(h, n_envs, 256, 8), 256, 0, stream, false,
                h->net, state, target_id, source_id, t, done_mask, step_ctr, env_offset, n_envs);
}

int pbn_unpack(pbn_handle* h, const uint64_t* state, void* out, int32_t out_kind, int64_t n_envs, void* stream_) {
  if (!h || !state || !out || n_envs < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  if (n_envs == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  const int grid = grid_for(h, n_envs * h->net.n_genes, 256, 8);
  if (out_kind == PBN_UNPACK_U8)
    return launch(h, unpack_kernel<uint8_t>, grid, 256, 0, stream, false, state, static_cast<uint8_t*>(out), h->net.n_genes, h->W, n_envs);
  if (out_kind == PBN_UNPACK_F32)
    return launch(h, unpack_kernel<float>, grid, 256, 0, stream, false, state, static_cast<float*>(out), h->net.n_genes, h->W, n_envs);
  return fail(PBN_ERR_INVALID, "out_kind=%d unknown", out_kind);
}

int pbn_advance_counter(pbn_handle* h, uint64_t* step_ctr_dev, uint64_t n, void* stream_) {
  if (!h || !step_ctr_dev) return fail(PBN_ERR_INVALID, "bad arguments");
  DeviceGuard guard(h->device);
  const int rc = launch(h, advance_counter_kernel, 1, 1, 0, static_cast<cudaStream_t>(stream_), false, step_ctr_dev, n);
  if (rc == PBN_OK) g_last_advance = h;
  return rc;
}

static int check_replay(const pbn_replay* r) {
  if (!r || r->capacity < 1 || !r->state || !r->next_state || !r->target_id || !r->actions || !r->reward || !r->done)
    return fail(PBN_ERR_INVALID, "replay ring: null array or capacity < 1");
  return PBN_OK;
}

int pbn_replay_observe(pbn_handle* h, const pbn_replay* r, int64_t head, const uint64_t* state, const int32_t* target_id,
                       int64_t n_envs, void* stream_) {
  if (!h || !state || n_envs < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  int rc = check_replay(r);
  if (rc != PBN_OK) return rc;
  if (head < 0 || head >= r->capacity || n_envs > r->capacity) return fail(PBN_ERR_INVALID, "replay push: head=%lld, n=%lld, capacity=%lld", (long long)head, (long long)n_envs, (long long)r->capacity);
  if (n_envs == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, replay_observe_kernel, grid_for(h, n_envs * h->W, 256, 8), 256, 0, stream, false, *r, head, state,
                target_id, h->W, n_envs);
}

int pbn_replay_commit(pbn_handle* h, const pbn_replay* r, int64_t head, const uint8_t* actions, const float* reward,
                      const uint8_t* terminated, const uint8_t* truncated, const uint64_t* next_state, int64_t n_envs,
                      void* stream_) {
  if (!h || !reward || !terminated || !next_state || n_envs < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  int rc = check_replay(r);
  if (rc != PBN_OK) return rc;
  if (head < 0 || head >= r->capacity || n_envs > r->capacity) return fail(PBN_ERR_INVALID, "replay push: head=%lld, n=%lld, capacity=%lld", (long long)head, (long long)n_envs, (long long)r->capacity);
  if (n_envs == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, replay_commit_kernel, grid_for(h, n_envs * h->net.bins, 256, 8), 256, 0, stream, false, *r, head,
                actions, reward, terminated, truncated, next_state, h->W, h->net.bins, n_envs);
}

int pbn_replay_sample(pbn_handle* h, const pbn_replay* r, const int64_t* index, int64_t batch, float* obs, float* next_obs,
                      int64_t* actions, float* reward, float* done, void* stream_) {
  if (!h || !index || batch < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  int rc = check_replay(r);
  if (rc != PBN_OK) return rc;
  if (batch == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  if ((obs || next_obs) &&
      (rc = launch(h, gather_unpack_kernel, grid_for(h, batch * h->net.n_genes, 256, 8), 256, 0, stream, false, h->net,
                   r->state, r->next_state, r->target_id, index, h->W, batch, obs, next_obs)) != PBN_OK)
    return rc;
  if (actions || reward || done)
    return launch(h, gather_scalars_kernel, grid_for(h, batch * h->net.bins, 256, 8), 256, 0, stream, false, *r, index,
                  h->net.bins, batch, actions, reward, done);
  return PBN_OK;
}

static int64_t per_leaves(int64_t capacity) {
  int64_t L = 1;
  while (L < capacity) L <<= 1;
  return L;
}

int64_t pbn_per_tree_floats(int64_t capacity) {
  if (capacity < 1 || capacity > (int64_t(1) << 30)) return fail(PBN_ERR_INVALID, "PER capacity=%lld outside 1..2^30", (long long)capacity);
  return 5 * per_leaves(capacity);
}

static int check_per(const pbn_handle* h, const pbn_per* p, PerView* v) {
  if (!h || !p || !p->tree || !p->max_p) return fail(PBN_ERR_INVALID, "PER: null argument");
  if (p->capacity < 1 || p->capacity > (int64_t(1) << 30)) return fail(PBN_ERR_INVALID, "PER capacity=%lld outside 1..2^30", (long long)p->capacity);
  if (!(p->alpha >= 0.0f) || std::isinf(p->alpha)) return fail(PBN_ERR_INVALID, "PER alpha=%g must be finite and >= 0", p->alpha);
  if (reinterpret_cast<uintptr_t>(p->tree) & 3u || reinterpret_cast<uintptr_t>(p->max_p) & 3u) return fail(PBN_ERR_INVALID, "PER arrays must be 4-byte aligned");
  v->L = per_leaves(p->capacity);
  v->D = 0;
  while ((int64_t(1) << v->D) < v->L) ++v->D;
  v->sum = p->tree;
  v->mn = p->tree + 2 * v->L;
  v->owner = reinterpret_cast<int*>(p->tree + 4 * v->L);
  v->ticket = reinterpret_cast<unsigned int*>(p->tree);
  v->max_p = p->max_p;
  v->capacity = p->capacity;
  v->alpha = p->alpha;
  return PBN_OK;
}

// One launch of the tile rebuild over slot ranges [a0, b0) and [a1, b1) (each tile of the grid exactly once).
static int per_rebuild(pbn_handle* h, const PerView& v, int64_t a0, int64_t b0, int64_t a1, int64_t b1, int fill,
                       const int64_t* reset_index, int64_t reset_n, cudaStream_t stream) {
  PerRanges r{};
  r.a0 = a0, r.b0 = b0, r.a1 = a1, r.b1 = b1, r.fill = fill;
  r.lt = std::min(v.D, kPerTileLog2);
  r.t0 = a0 >> r.lt;
  r.n0 = ((b0 - 1) >> r.lt) - r.t0 + 1;
  int64_t t1_end = b1 > a1 ? ((b1 - 1) >> r.lt) + 1 : 0;
  r.t1 = a1 >> r.lt;
  if (t1_end > r.t0) t1_end = r.t0;   // a tile the first range already covers
  const int64_t n1 = std::max<int64_t>(0, t1_end - r.t1);
  return launch(h, per_rebuild_kernel, (unsigned)(r.n0 + n1), kPerRebuildThreads, 0, stream, false, v, r, reset_index,
                reset_n);
}

int pbn_per_init(pbn_handle* h, const pbn_per* p, void* stream_) {
  PerView v;
  int rc = check_per(h, p, &v);
  if (rc != PBN_OK) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, per_init_kernel, grid_for(h, 2 * v.L, 256, 8), 256, 0, stream, false, v);
}

int pbn_per_push(pbn_handle* h, const pbn_per* p, int64_t head, int64_t n, void* stream_) {
  PerView v;
  int rc = check_per(h, p, &v);
  if (rc != PBN_OK) return rc;
  if (head < 0 || head >= p->capacity || n < 0 || n > p->capacity) return fail(PBN_ERR_INVALID, "PER push: head=%lld, n=%lld, capacity=%lld", (long long)head, (long long)n, (long long)p->capacity);
  if (n == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  const int64_t end = head + n;
  if (end <= p->capacity) return per_rebuild(h, v, head, end, 0, 0, 1, nullptr, 0, stream);
  return per_rebuild(h, v, head, p->capacity, 0, end - p->capacity, 1, nullptr, 0, stream);
}

int pbn_per_update(pbn_handle* h, const pbn_per* p, const int64_t* index, const float* td_error, int64_t batch, float eps,
                   void* stream_) {
  PerView v;
  int rc = check_per(h, p, &v);
  if (rc != PBN_OK) return rc;
  if (!index || !td_error || batch < 0 || batch > 0x7FFFFFFF) return fail(PBN_ERR_INVALID, "bad arguments");
  if (!(eps > 0.0f) || std::isinf(eps)) return fail(PBN_ERR_INVALID, "PER eps=%g must be finite and > 0", eps);
  if (batch == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  if (batch <= kPerUpdateOneCta)
    return launch(h, per_update_cta_kernel, 1, kPerUpdateThreads, 0, stream, false, v, index, td_error, (int)batch, eps);
  const int grid = grid_for(h, batch, 256, 8);
  if ((rc = launch(h, per_update_claim_kernel, grid, 256, 0, stream, false, v, index, batch)) != PBN_OK ||
      (rc = launch(h, per_update_write_kernel, grid, 256, 0, stream, false, v, index, td_error, batch, eps)) != PBN_OK)
    return rc;
  return per_rebuild(h, v, 0, v.L, 0, 0, 0, index, batch, stream);
}

int pbn_per_sample(pbn_handle* h, const pbn_per* p, const float* u, int64_t batch, float beta, int64_t* index,
                   float* weight, void* stream_) {
  PerView v;
  int rc = check_per(h, p, &v);
  if (rc != PBN_OK) return rc;
  if (!u || !index || !weight || batch < 0 || batch > (int64_t(1) << 24)) return fail(PBN_ERR_INVALID, "bad arguments");
  if (!(beta >= 0.0f) || std::isinf(beta)) return fail(PBN_ERR_INVALID, "PER beta=%g must be finite and >= 0", beta);
  if (batch == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, per_sample_kernel, grid_for(h, batch * 32, 256, 8), 256, 0, stream, false, v, u, batch, beta, index,
                weight);
}

int pbn_observe(pbn_handle* h, const uint64_t* state, const int32_t* target_id, float* obs, int64_t n_envs, void* stream_) {
  if (!h || !state || !obs || n_envs < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  if (n_envs == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, gather_unpack_kernel, grid_for(h, n_envs * h->net.n_genes, 256, 8), 256, 0, stream, false, h->net,
                state, nullptr, target_id, nullptr, h->W, n_envs, obs, nullptr);
}

int pbn_in_target(pbn_handle* h, const uint64_t* state, const int32_t* target_id, uint8_t* out, int64_t n_envs, void* stream_) {
  if (!h || !state || !target_id || !out || n_envs < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  if (n_envs == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, h->W == 1 ? in_target_kernel<1> : in_target_kernel<2>, grid_for(h, n_envs, 256, 8), 256, 0, stream,
                false, h->net, state, target_id, out, n_envs);
}

int pbn_rollout_track(pbn_handle* h, const uint8_t* terminated, uint8_t* active, int32_t* count, int32_t max_steps,
                      int64_t n_envs, unsigned int* n_active, void* stream_) {
  if (!h || !terminated || !active || !count || n_envs < 0 || max_steps < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  if (n_envs == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, rollout_track_kernel, grid_for(h, n_envs, 256, 8), 256, 0, stream, false, terminated, active, count,
                max_steps, n_envs, n_active);
}

int pbn_rollout_reduce(pbn_handle* h, const int32_t* count, const int32_t* pair_id, int64_t n_envs, int32_t n_pairs,
                       int32_t max_steps, unsigned long long* matrix, unsigned long long* hist, void* stream_) {
  if (!h || !count || !pair_id || !matrix || !hist || n_envs < 0 || n_pairs < 1 || max_steps < 0)
    return fail(PBN_ERR_INVALID, "bad arguments");
  if (n_envs == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, rollout_reduce_kernel, grid_for(h, n_envs, 256, 8), 256, 0, stream, false, count, pair_id, n_envs,
                n_pairs, max_steps, matrix, hist);
}

int pbn_visit_count(pbn_handle* h, const uint64_t* state, const uint8_t* mask, int64_t n_envs, unsigned long long* tags,
                    uint64_t* slot_state, unsigned long long* counts, int64_t capacity, unsigned int* overflow, void* stream_) {
  if (!h || !state || !tags || !slot_state || !counts || !overflow || n_envs < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  if (capacity < 2 || (capacity & (capacity - 1))) return fail(PBN_ERR_INVALID, "capacity=%lld must be a power of two >= 2", (long long)capacity);
  if (n_envs == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, h->W == 1 ? visit_count_kernel<1> : visit_count_kernel<2>, grid_for(h, n_envs, 256, 8), 256, 0, stream,
                false, state, mask, n_envs, tags, slot_state, counts, (uint64_t)capacity - 1,
                h->W == 1 && h->net.n_genes <= 63, overflow);
}

int pbn_successor_sets(pbn_handle* h, const uint64_t* state, int64_t n_states, uint64_t* can1, uint64_t* can0, void* stream_) {
  if (!h || !state || !can1 || !can0 || n_states < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  if (n_states == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, h->W == 1 ? successor_sets_kernel<1> : successor_sets_kernel<2>, grid_for(h, n_states, 256, 8), 256, 0,
                stream, false, h->net, state, n_states, can1, can0);
}

int pbn_closure_expand(pbn_handle* h, uint64_t* list, int64_t begin, int64_t end, int64_t list_cap, unsigned long long* list_count,
                       unsigned long long* tags, uint64_t* slot_state, unsigned long long* slot_index, int64_t capacity,
                       int32_t max_free, int32_t* status, void* stream_) {
  if (!h || !list || !list_count || !tags || !slot_state || !slot_index || !status || begin < 0 || end < begin || end > list_cap)
    return fail(PBN_ERR_INVALID, "bad arguments");
  if (capacity < 2 || (capacity & (capacity - 1))) return fail(PBN_ERR_INVALID, "capacity=%lld must be a power of two >= 2", (long long)capacity);
  if (max_free < 0 || max_free > kClosureMaxFree) return fail(PBN_ERR_INVALID, "max_free=%d outside 0..%d", max_free, kClosureMaxFree);
  if (end == begin) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, h->W == 1 ? closure_expand_kernel<1> : closure_expand_kernel<2>, grid_for(h, (end - begin) * 128, 128, 16),
                128, 0, stream, false, h->net, list, begin, end, list_cap, list_count, tags, slot_state, slot_index,
                (uint64_t)capacity - 1, max_free, status);
}

int pbn_closure_reach(pbn_handle* h, const uint64_t* list, int64_t count, uint8_t* flags, const unsigned long long* tags,
                      const uint64_t* slot_state, const unsigned long long* slot_index, int64_t capacity, int32_t* changed,
                      void* stream_) {
  if (!h || !list || !flags || !tags || !slot_state || !slot_index || !changed || count < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  if (capacity < 2 || (capacity & (capacity - 1))) return fail(PBN_ERR_INVALID, "capacity=%lld must be a power of two >= 2", (long long)capacity);
  if (count == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, h->W == 1 ? closure_reach_kernel<1> : closure_reach_kernel<2>, grid_for(h, count * 128, 128, 16), 128, 0,
                stream, false, h->net, list, count, flags, tags, slot_state, slot_index, (uint64_t)capacity - 1, changed);
}

int64_t pbn_resident_words(const pbn_handle* h, int64_t n_envs) {
  if (!h || n_envs < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  const int64_t tiles = (n_envs + 1023) / 1024;
  const int64_t nt = tiles > 0 ? tiles : 1;
  return nt * 32 * (int64_t)resident_rows(h->net.n_genes) + ((nt + 31) / 32) * 32;   // + one epoch word per tile
}

int pbn_resident_import(pbn_handle* h, uint32_t* resident, const uint64_t* state, const int32_t* target_id, const uint16_t* t,
                        int64_t n_envs, void* stream_) {
  if (!h || !resident || !state || n_envs < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  int rc = resident_supported(h);
  if (rc != PBN_OK) return rc;
  if (n_envs == 0) return PBN_OK;
  if (target_id && h->net.n_attr == 0) return fail(PBN_ERR_NO_ATTRACTORS, "target_id given but no attractor table uploaded");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  const int64_t nt = (n_envs + 1023) / 1024;
  if ((rc = launch(h, h->W == 1 ? resident_import_kernel<1> : resident_import_kernel<2>, grid_for(h, nt * 1024, 256, 8), 256,
                   0, stream, false, h->net, resident, state, target_id, t, n_envs)) != PBN_OK)
    return rc;
  PBN_CUDA(cudaMemsetAsync(resident + nt * 32 * (int64_t)resident_rows(h->net.n_genes), 0, (size_t)((nt + 31) / 32) * 32 * 4, stream));
  return PBN_OK;
}

int pbn_resident_export(pbn_handle* h, const uint32_t* resident, uint64_t* state, int32_t* target_id, uint16_t* t,
                        int64_t n_envs, void* stream_) {
  if (!h || !resident || n_envs < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  if (n_envs == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, h->W == 1 ? resident_export_kernel<1> : resident_export_kernel<2>,
                grid_for(h, ((n_envs + 1023) / 1024) * 1024, 256, 8), 256, 0, stream, false, h->net, resident, state, target_id,
                t, n_envs);
}

int pbn_pack(pbn_handle* h, const uint8_t* bits, uint64_t* state, int64_t n_envs, void* stream_) {
  if (!h || !state || !bits || n_envs < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  if (n_envs == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, pack_kernel, grid_for(h, n_envs * h->W, 256, 8), 256, 0, stream, false, bits, state, h->net.n_genes,
                h->W, n_envs);
}

int pbn_attractor_id(pbn_handle* h, const uint64_t* state, int32_t* attr_id, int64_t n_envs, void* stream_) {
  if (!h || !state || !attr_id || n_envs < 0) return fail(PBN_ERR_INVALID, "bad arguments");
  if (n_envs == 0) return PBN_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  return launch(h, h->W == 1 ? attractor_id_kernel<1> : attractor_id_kernel<2>, grid_for(h, n_envs, 256, 8), 256, 0, stream,
                false, h->net, state, attr_id, n_envs);
}

// ---- exact optimal control (control.cuh) ----
static constexpr uint32_t kDpSliceStates = 1u << 22;   // states (or state pairs) per launch

// The perturbation model a backup applies: PBN_PERT_NONE whenever p = 0; model C with p > 0 is refused.
static int dp_model(const pbn_handle* h, const char* who, int* model) {
  if (!h) return fail(PBN_ERR_INVALID, "%s: null handle", who);
  if (h->net.n_genes > PBN_DP_MAX_GENES)
    return fail(PBN_ERR_UNSUPPORTED, "%s: %d genes, exact control covers at most %d", who, h->net.n_genes, PBN_DP_MAX_GENES);
  *model = h->perturb_p > 0.0 ? h->net.pert_mode : PBN_PERT_NONE;
  if (*model == PBN_PERT_C)
    return fail(PBN_ERR_UNSUPPORTED, "%s: perturbation model C with p > 0 makes every gene free (a backup of O(4^N))", who);
  return PBN_OK;
}

int64_t pbn_dp_workspace_bytes(const pbn_handle* h) {
  int model, rc;
  if ((rc = dp_model(h, "pbn_dp_workspace_bytes", &model)) != PBN_OK) return rc;
  return (int64_t)24 << h->net.n_genes;   // two (fp64 value, u32 endpoint) buffers of the relaxation; expect uses the first
}

// out = K_p in over all 2^N states: the low genes tile by tile in shared memory, then one in-place pass per higher gene.
static int dp_kp(pbn_handle* h, const double* in, double* out, cudaStream_t stream) {
  const int N = h->net.n_genes;
  const uint32_t S = 1u << N;
  const double p = h->perturb_p;
  const int tb = N < kKpTileBits ? N : kKpTileBits;
  const uint32_t tiles = S >> tb, per = kDpSliceStates >> tb;
  int rc;
  for (uint32_t t0 = 0; t0 < tiles; t0 += per) {
    const uint32_t nt = tiles - t0 < per ? tiles - t0 : per;
    if ((rc = launch(h, dp_kp_low_kernel, grid_for(h, (int64_t)nt * 256, 256, 8), 256, 0, stream, false, in, out, tb,
                     t0, nt, p)) != PBN_OK)
      return rc;
  }
  for (int b = tb; b < N; ++b)
    for (uint32_t j0 = 0; j0 < S / 2; j0 += kDpSliceStates) {
      const uint32_t cnt = S / 2 - j0 < kDpSliceStates ? S / 2 - j0 : kDpSliceStates;
      if ((rc = launch(h, dp_kp_bit_kernel, grid_for(h, cnt, 256, 8), 256, 0, stream, false, out, b, j0, cnt, p)) != PBN_OK)
        return rc;
    }
  return PBN_OK;
}

int pbn_dp_expect(pbn_handle* h, const double* func_prob, const double* u_in, double* w, void* workspace, void* stream_) {
  int model, rc;
  if ((rc = dp_model(h, "pbn_dp_expect", &model)) != PBN_OK) return rc;
  if (!func_prob || !u_in || !w) return fail(PBN_ERR_INVALID, "pbn_dp_expect: null array");
  if (u_in == w) return fail(PBN_ERR_INVALID, "pbn_dp_expect: w must not alias u_in");
  if (model != PBN_PERT_NONE && !workspace) return fail(PBN_ERR_INVALID, "pbn_dp_expect: perturbation needs the workspace");
  const int N = h->net.n_genes;
  const uint32_t S = 1u << N;
  const double p = h->perturb_p;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  double* kpu = static_cast<double*>(workspace);
  if (model != PBN_PERT_NONE && (rc = dp_kp(h, u_in, kpu, stream)) != PBN_OK) return rc;
  const double c = std::pow(1.0 - p, (double)N);
  for (uint32_t s0 = 0; s0 < S; s0 += kDpSliceStates) {
    const uint32_t cnt = S - s0 < kDpSliceStates ? S - s0 : kDpSliceStates;
    if ((rc = launch(h, dp_expect_kernel, grid_for(h, (int64_t)cnt * 32, kDpWarps * 32, 8), kDpWarps * 32, 0, stream, false,
                     h->net, func_prob, model == PBN_PERT_B ? kpu : u_in, w, s0, cnt)) != PBN_OK)
      return rc;
    if (model == PBN_PERT_A &&
        (rc = launch(h, dp_mix_kernel, grid_for(h, cnt, 256, 8), 256, 0, stream, false, w, kpu, u_in, c, s0, cnt)) != PBN_OK)
      return rc;
  }
  return PBN_OK;
}

// acc (2^N u64 fixed-point units) -> fp64 in place.
static int dp_fix(pbn_handle* h, unsigned long long* acc, cudaStream_t stream) {
  const uint32_t S = 1u << h->net.n_genes;
  for (uint32_t s0 = 0; s0 < S; s0 += kDpSliceStates) {
    const uint32_t cnt = S - s0 < kDpSliceStates ? S - s0 : kDpSliceStates;
    const int rc = launch(h, dp_fix_kernel, grid_for(h, cnt, 256, 8), 256, 0, stream, false, acc, s0, cnt);
    if (rc != PBN_OK) return rc;
  }
  return PBN_OK;
}

// The forward operator, by the transposes of expect's steps (K_p is symmetric):
//   NONE: y = x' F;   B: y = (x' F) K_p;   A: y = c (x' F) + x' K_p - c x',   x' = x M_mu (masks) or x.
// Workspace: [0, 2^N) holds x M_mu, [2^N, 2^(N+1)) the push of model B or x' K_p of model A.
int pbn_dp_push(pbn_handle* h, const double* func_prob, const double* x_in, const uint32_t* masks, double* y,
                void* workspace, void* stream_) {
  int model, rc;
  if ((rc = dp_model(h, "pbn_dp_push", &model)) != PBN_OK) return rc;
  if (!func_prob || !x_in || !y) return fail(PBN_ERR_INVALID, "pbn_dp_push: null array");
  if (x_in == y) return fail(PBN_ERR_INVALID, "pbn_dp_push: y must not alias x_in");
  if ((model != PBN_PERT_NONE || masks) && !workspace)
    return fail(PBN_ERR_INVALID, "pbn_dp_push: perturbation or masks need the workspace");
  const int N = h->net.n_genes;
  const uint32_t S = 1u << N;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  double* ws = static_cast<double*>(workspace);
  double* second = ws ? ws + S : nullptr;
  const double* src = x_in;
  if (masks) {
    unsigned long long* acc = reinterpret_cast<unsigned long long*>(ws);
    PBN_CUDA(cudaMemsetAsync(acc, 0, (size_t)S * sizeof(double), stream));
    for (uint32_t s0 = 0; s0 < S; s0 += kDpSliceStates) {
      const uint32_t cnt = S - s0 < kDpSliceStates ? S - s0 : kDpSliceStates;
      if ((rc = launch(h, dp_flip_push_kernel, grid_for(h, cnt, 256, 8), 256, 0, stream, false, x_in, masks, acc, S - 1u,
                       s0, cnt)) != PBN_OK)
        return rc;
    }
    if ((rc = dp_fix(h, acc, stream)) != PBN_OK) return rc;
    src = ws;
  }
  if (model == PBN_PERT_A && (rc = dp_kp(h, src, second, stream)) != PBN_OK) return rc;
  unsigned long long* acc = reinterpret_cast<unsigned long long*>(model == PBN_PERT_B ? second : y);
  PBN_CUDA(cudaMemsetAsync(acc, 0, (size_t)S * sizeof(double), stream));
  for (uint32_t s0 = 0; s0 < S; s0 += kDpSliceStates) {
    const uint32_t cnt = S - s0 < kDpSliceStates ? S - s0 : kDpSliceStates;
    if ((rc = launch(h, dp_push_kernel, grid_for(h, (int64_t)cnt * 32, kDpWarps * 32, 8), kDpWarps * 32, 0, stream, false,
                     h->net, func_prob, src, acc, s0, cnt)) != PBN_OK)
      return rc;
  }
  if ((rc = dp_fix(h, acc, stream)) != PBN_OK) return rc;
  if (model == PBN_PERT_B) return dp_kp(h, second, y, stream);
  if (model == PBN_PERT_A) {
    const double c = std::pow(1.0 - h->perturb_p, (double)N);
    for (uint32_t s0 = 0; s0 < S; s0 += kDpSliceStates) {
      const uint32_t cnt = S - s0 < kDpSliceStates ? S - s0 : kDpSliceStates;
      if ((rc = launch(h, dp_mix_kernel, grid_for(h, cnt, 256, 8), 256, 0, stream, false, y, second, src, c, s0, cnt)) !=
          PBN_OK)
        return rc;
    }
  }
  return PBN_OK;
}

int pbn_dp_improve(pbn_handle* h, const double* w, uint64_t flip_genes, int32_t max_flips, double r_action, double* v,
                   uint32_t* policy, void* workspace, void* stream_) {
  if (!h) return fail(PBN_ERR_INVALID, "pbn_dp_improve: null handle");
  const int N = h->net.n_genes;
  if (N > PBN_DP_MAX_GENES)
    return fail(PBN_ERR_UNSUPPORTED, "pbn_dp_improve: %d genes, exact control covers at most %d", N, PBN_DP_MAX_GENES);
  if (!w || !v) return fail(PBN_ERR_INVALID, "pbn_dp_improve: null array");
  if (w == v) return fail(PBN_ERR_INVALID, "pbn_dp_improve: v must not alias w");
  if (!(r_action <= 0.0)) return fail(PBN_ERR_INVALID, "pbn_dp_improve: r_action=%g must be <= 0", r_action);
  if (max_flips < 0 || max_flips > PBN_MAX_BINS) return fail(PBN_ERR_INVALID, "pbn_dp_improve: max_flips=%d outside 0..%d", max_flips, PBN_MAX_BINS);
  if (flip_genes >> N) return fail(PBN_ERR_INVALID, "pbn_dp_improve: flip_genes has genes beyond the %d of the network", N);
  if (max_flips >= 2 && !workspace) return fail(PBN_ERR_INVALID, "pbn_dp_improve: max_flips >= 2 needs the workspace");
  const uint32_t S = 1u << N;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  // ping-pong buffers of the relaxation: values [2][S] fp64, then endpoints [2][S] u32
  double* bv[2] = {static_cast<double*>(workspace), workspace ? static_cast<double*>(workspace) + S : nullptr};
  uint32_t* be[2] = {workspace ? reinterpret_cast<uint32_t*>(static_cast<double*>(workspace) + 2 * (size_t)S) : nullptr,
                     workspace ? reinterpret_cast<uint32_t*>(static_cast<double*>(workspace) + 2 * (size_t)S) + S : nullptr};
  const double cost0 = r_action * 0.0;
  for (int k = max_flips == 0 ? 0 : 1; k <= max_flips; ++k) {
    const double* ival = k >= 2 ? bv[k & 1] : nullptr;        // B_{k-1}: w itself for k = 1
    const uint32_t* iend = k >= 2 ? be[k & 1] : nullptr;
    double* oval = k < max_flips ? bv[(k + 1) & 1] : nullptr;  // B_k, unless this is the last pass
    uint32_t* oend = k < max_flips ? be[(k + 1) & 1] : nullptr;
    const double cost_k = r_action * (double)k;
    for (uint32_t s0 = 0; s0 < S; s0 += kDpSliceStates) {
      const uint32_t cnt = S - s0 < kDpSliceStates ? S - s0 : kDpSliceStates;
      const int rc = launch(h, dp_improve_kernel, grid_for(h, cnt, 256, 8), 256, 0, stream, false, w, ival, iend, oval, oend,
                            v, policy, (uint32_t)flip_genes, k, cost0, cost_k, s0, cnt);
      if (rc != PBN_OK) return rc;
    }
  }
  return PBN_OK;
}

}  // extern "C"
