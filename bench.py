#!/usr/bin/env python
"""PBN env-steps/s benchmark (BASELINE.json metric): Bittner-28, 2^20 env instances per GPU.

    python bench.py --gpus 1 --steps K --warmup W               # this repo's CUDA path
    python bench.py --impl reference --gpus 1 --steps K --warmup W   # CPU arm (oracle port on host cores)
    torchrun ... bench.py --gpus N ...                           # one rank per GPU, weak scaling
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # also write the last timed step's results

The benchmark writes nothing into the source tree (which may be read-only): network specialisations that
build() did not compile are cached in a temporary directory for the run.

A "step" is one pbn_step launch over one batch of 2^20 env instances (per GPU): apply the
agent's gene flips, draw predictor selections + perturbations from Philox, synchronous
Boolean update, target-attractor test, reward/done, auto-reset.  Prints ONE JSON line.

Timing: steps are captured into a CUDA graph (the launch-bound inner loop; the Philox step
counter lives in device memory so every replay advances the streams) and replayed; the launches use
programmatic dependent launch, so a step draws its state-independent predictor-selection planes
while the previous kernel drains and only then waits for it; the timed
region is bracketed by barrier + torch.cuda.synchronize() and CUDA events on the launching
stream; max over ranks.  The L2 (126 MB) is defeated by rotating over R independent env
batches whose combined working set exceeds it, plus a pool of distinct action buffers.
"""
import argparse
import atexit
import json
import os
import shutil
import sys
import tempfile
import threading
import time
from pathlib import Path

sys.dont_write_bytecode = True   # no __pycache__ in the source tree
ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

GOLD = ROOT / "tests" / "golden"
METRIC = "PBN env-steps/sec (Bittner-28, 2^20 envs) at 1/2/4/8 B200 vs host CPU"
UNIT = "env-steps/s"
BYTES_PER_STEP = {1: 33, 2: 49}  # algorithmic HBM bytes per env-step by words/state (SURVEY.md 8d)


# ----------------------------------------------------------------------------------------------
# workload
# ----------------------------------------------------------------------------------------------

def load_workload(name):
    """Network + attractor/target table for a golden network (same choices as tests/helpers.py)."""
    import numpy as np
    from pbn_rl_b200 import AttractorSet, PBNNetwork, sorted_id_permutation
    net = PBNNetwork.from_json(GOLD / f"{name}.json")
    if name == "pbn28":
        raw = json.loads((GOLD / "attractors_bittner28.json").read_text())["attractors"]
        attrs = AttractorSet([[tuple(s) for s in a] for a in raw], 28).permuted(sorted_id_permutation(net.genes))
    elif name == "pbn7":
        raw = json.loads((GOLD / "attractors_bittner7.json").read_text())["attractors"]
        attrs = AttractorSet([[tuple(s) for s in a] for a in raw], 7)
    elif name == "pbn10":
        sinks = json.loads((GOLD / "k5_stg.json").read_text())["pbn10"]["sink_sccs"]
        attrs = AttractorSet([[tuple((s >> i) & 1 for i in range(10)) for s in m] for m in sinks], 10)
    else:
        rng = np.random.default_rng(70)
        states = rng.integers(0, 2, size=(16, net.n_genes))
        attrs = AttractorSet([[tuple(int(v) for v in s)] for s in states], net.n_genes)
    return net, attrs


ENV_KW = dict(horizon=20, bins=3, perturb_p=0.001, perturb_mode="A", r_success=5.0, r_step=0.0, r_action=-1.0,
              seed=0x5EED)


def use_private_jit_cache():
    """Point the library's cubin cache (PBN_B200_CACHE) at a temporary directory that links the cubins build() left in
    pbn_rl_b200/_jit_cache/, so that specialisations compiled at run time land there and not in the source tree.
    The directory is removed at exit.  An explicit PBN_B200_CACHE is left alone."""
    if os.environ.get("PBN_B200_CACHE"):
        return
    tmp = tempfile.mkdtemp(prefix="pbn_b200_cache_")
    atexit.register(shutil.rmtree, tmp, True)
    for cubin in (ROOT / "pbn_rl_b200" / "_jit_cache").glob("*.cubin"):
        os.symlink(cubin, os.path.join(tmp, cubin.name))
    os.environ["PBN_B200_CACHE"] = tmp


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------

class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index, period=0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                bits = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle's per-instance env on the host cores
# ----------------------------------------------------------------------------------------------

_CPU_ENV = {}


def _cpu_env(name, seed):
    """Per-process cached oracle env (built once per worker process)."""
    key = (name, seed)
    if key not in _CPU_ENV:
        import numpy as np
        from oracle import pbn_oracle as O
        onet = O.OracleNetwork.from_json(GOLD / f"{name}.json")
        _, attrs = load_workload(name)
        env = O.OraclePBNEnv(onet, attrs.attractors, horizon=ENV_KW["horizon"], perturb_p=ENV_KW["perturb_p"],
                             perturb_mode=ENV_KW["perturb_mode"], r_success=ENV_KW["r_success"],
                             r_step=ENV_KW["r_step"], r_action=ENV_KW["r_action"], seed=seed)
        env.reset()
        acts = np.random.default_rng(seed).integers(0, onet.n + 1, size=(4096, 3)).tolist()
        _CPU_ENV[key] = (env, acts)
    return _CPU_ENV[key]


def _cpu_worker(args):
    """Step one single-instance oracle env `n_steps` times (or for `seconds`) with random actions."""
    name, seed, n_steps, seconds = args
    env, acts = _cpu_env(name, seed)
    chunk = 64
    done_steps = 0
    t0 = time.perf_counter()
    while True:
        for i in range(chunk):
            _, _, term, trunc, _ = env.step(acts[(done_steps + i) & 4095])
            if term or trunc:
                env.reset()
        done_steps += chunk
        if n_steps is not None and done_steps >= n_steps:
            break
        if seconds is not None and time.perf_counter() - t0 >= seconds:
            break
    return done_steps, time.perf_counter() - t0


class CpuArm:
    """`cores` worker processes, one oracle env each; run() = one bounded sample on all of them."""

    def __init__(self, name, cores):
        import multiprocessing as mp
        self.name, self.cores = name, cores
        self.pool = mp.get_context("fork").Pool(cores) if cores > 1 else None

    def run(self, n_steps=None, seconds=None):
        jobs = [(self.name, 1000 + i, n_steps, seconds) for i in range(self.cores)]
        res = self.pool.map(_cpu_worker, jobs, chunksize=1) if self.pool else [_cpu_worker(jobs[0])]
        return sum(r[0] for r in res), max(max(r[1] for r in res), 1e-9)

    def close(self):
        if self.pool:
            self.pool.close()
            self.pool.join()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    K, Wm = args.steps_ref, args.warmup_ref
    # bounded sample per bench "step", sized so K + W steps take about a minute of wall clock
    # (the per-instance python env does roughly 2e4 env-steps/s per core)
    per_proc = int(min(4096, max(64, (60.0 * 2.0e4) / max(K + Wm, 1))) // 64 * 64)
    arm = CpuArm(args.net, cores)
    for _ in range(Wm):
        arm.run(n_steps=per_proc)
    total, busy = 0, 0.0
    for _ in range(K):
        n, t = arm.run(n_steps=per_proc)
        total += n
        busy += t
    arm.close()
    value = total / busy
    sample = ("%d processes x %d env-steps per bench step (a bounded sample of the 2^20-env workload: ms_per_step of this arm is "
              "the time of that sample, not of 2^20 env-steps; the rate is what compares), single-env oracle port, %s"
              % (cores, per_proc, args.net))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": K, "warmup": Wm, "ms_per_step": 1e3 * busy / max(K, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args, int(os.environ.get("WORLD_SIZE", "1")), None),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------

def workload_config(args, world, kernel):
    return {
        "workload": "Bittner-28 PBN (kaban/pbn28.ispl, data/attractors_Bittner-28.pkl), 2^20 env instances per GPU"
        if args.net == "pbn28" and args.envs == 1 << 20 else "%s, %d env instances per GPU" % (args.net, args.envs),
        "network": args.net, "envs_per_gpu": args.envs, "total_envs": args.envs * world, "bins": 3,
        "horizon": 20, "perturb_p": 0.001, "perturb_mode": "A", "auto_reset": True,
        "actions": "uniform in [0,N], pre-generated on device, pool of %d buffers" % args.action_pool,
        "l2": "%d rotating env batches + action pool: working set > 126 MB L2, no flush" % args.batches,
        "graph_steps": min(args.graph_steps, max(1, args.steps or 1)), "kernel": kernel,
        "launch": "CUDA graph of %d step launches%s" % (min(args.graph_steps, max(1, args.steps or 1)), "" if getattr(args, "no_pdl", False) else
                                                        ", programmatic dependent launch (selection planes drawn under the previous kernel's tail)"), "parallelism": "env-sharded x%d" % world,
        "state_layout": "plane-resident (pbn_step with args->resident%s)" % (", tile-chained launches" if getattr(args, "chain", False) else "")
        if getattr(args, "resident", False) or getattr(args, "chain", False) else "row-format u64 words",
    }


def make_env(net, attrs, args, device, env_offset, device_counter=True, n_envs=None, resident=None, chain=None):
    import torch
    from pbn_rl_b200 import VecPBNEnv
    e = args.envs if n_envs is None else n_envs
    resident = (args.resident or args.chain) if resident is None else resident
    chain = args.chain if chain is None else chain
    env = VecPBNEnv(net, e, attrs, device=device, env_offset=env_offset, auto_reset=True,
                    device_counter=device_counter, pdl=not args.no_pdl, kernel=args.kernel, resident=resident, chain=chain, **ENV_KW)
    g = torch.Generator(device=device).manual_seed(env_offset + 1)
    n = net.n_genes
    st = env.state
    for w in range(net.n_words):
        bits = min(64, n - 64 * w)
        hi = torch.randint(0, 1 << max(bits - 31, 0), (e,), generator=g, device=device, dtype=torch.int64)
        lo = torch.randint(0, 1 << min(bits, 31), (e,), generator=g, device=device, dtype=torch.int64)
        st[:, w] = (hi << 31) | lo
    env.set_target(torch.randint(0, len(attrs), (e,), generator=g, device=device, dtype=torch.int32))
    return env


def time_steps(envs, pool, K, G, Wm, stream, world):
    """EXACTLY K timed step launches (K // G replays of a G-step CUDA graph + one tail graph) after Wm warm-up steps;
    barrier + synchronize on both sides, CUDA events on the launching stream.  Returns milliseconds (this rank)."""
    import torch
    import torch.distributed as dist
    R = len(envs)
    tail_steps = K % G

    def enqueue(i):
        envs[i % R].step(pool[i % len(pool)])

    with torch.cuda.stream(stream):
        for i in range(Wm):
            enqueue(i)
        for e in envs:
            e.advance_counter()
        stream.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            for i in range(G):
                enqueue(i)
            for e in envs:
                e.advance_counter()   # PDL launches do not bump the device step counter themselves
        graph.replay()
        tail = None
        if tail_steps:
            tail = torch.cuda.CUDAGraph()
            with torch.cuda.graph(tail, stream=stream):
                for i in range(tail_steps):
                    enqueue(i)
                for e in envs:
                    e.advance_counter()
            tail.replay()
        stream.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(K // G):
            graph.replay()
        if tail is not None:
            tail.replay()
        ev1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return ev0.elapsed_time(ev1)


DUMP_BYTES = 64 << 20


def dump_outputs(env, out_dir):
    """Write what the last timed step returned to its caller, for the env batch it stepped, as DIR/<name>.npy:
    state_u32 (float64 [E, 2W]: each int64 state word as its low and high 32-bit halves, exact in float64), reward,
    terminated and truncated (float32 [E]).  A batch whose arrays exceed 64 MB is cut to a fixed seeded sample of envs;
    env_index (float64) then lists the envs kept."""
    import numpy as np
    words = env.state.cpu().numpy().view(np.uint64)
    e = words.shape[0]
    out = {"state_u32": np.stack([words & 0xFFFFFFFF, words >> 32], axis=-1).reshape(e, -1).astype(np.float64),
           "reward": env.reward.cpu().numpy().astype(np.float32),
           "terminated": env.terminated.cpu().numpy().astype(np.float32),
           "truncated": env.truncated.cpu().numpy().astype(np.float32)}
    per_env = sum(a.nbytes for a in out.values()) // e
    if per_env * e > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(e, size=DUMP_BYTES // (per_env + 8), replace=False))
        out = {k: a[keep] for k, a in out.items()}
        out["env_index"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def max_over_ranks(ms, device, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_gpu(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    net, attrs = load_workload(args.net)
    W = net.n_words

    from pbn_rl_b200.dist import bind_to_gpu_numa
    affinity0 = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local_rank, rank=rank, world=world)   # before any page-locked allocation

    # R independent env batches (each `envs` instances); batch b of rank r owns global env ids
    # [(r*R + b) * envs, ...): disjoint Philox streams everywhere.
    R = args.batches
    envs = [make_env(net, attrs, args, device, (rank * R + b) * args.envs) for b in range(R)]
    g = torch.Generator(device=device).manual_seed(1234 + rank)
    pool = [torch.randint(0, net.n_genes + 1, (args.envs, 3), generator=g, device=device, dtype=torch.uint8)
            for _ in range(args.action_pool)]
    kernel = envs[0].kernel

    K = max(1, args.steps)                     # EXACTLY K timed steps
    G = min(args.graph_steps, K)
    Wm = max(3, args.warmup)
    stream = torch.cuda.Stream(device)
    stats_total = torch.zeros(8, dtype=torch.int64, device=device)

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms = time_steps(envs, pool, K, G, Wm, stream, world)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # every replay restarts the step index at 0: the last timed step is step (K % G or G) - 1 of its graph
        dump_outputs(envs[((K % G or G) - 1) % R], args.dump_outputs)

    # episode statistics: the only cross-GPU exchange of the path (one small NCCL all-reduce)
    for e in envs:
        stats_total += e.stats_buf
    if world > 1:
        dist.all_reduce(stats_total, op=dist.ReduceOp.SUM)
    ms = max_over_ranks(ms, device, world)
    value = args.envs * world * K / (ms * 1e-3)
    ms_per_step = ms / K
    bytes_per = BYTES_PER_STEP[W]
    achieved = bytes_per * args.envs / (ms_per_step * 1e-3) / 1e9
    peaks_file = ROOT / "MEASURED_PEAKS.json"
    if peaks_file.exists():
        peak, peak_src = float(json.loads(peaks_file.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"

    # BASELINE config 3 as written ("2^20 envs sharded over 1/2/4/8 B200"): the SAME total batch cut over the ranks,
    # envs / world instances per GPU (strong scaling); efficiency = this value / the weak-scaling value above, whose
    # per-rank work is the whole batch
    strong = None
    if world > 1 or args.strong:
        per = max(1024, (args.envs // world) // 1024 * 1024)
        # small per-GPU batches (below 2 tiles per SM and CTA slot) are latency-bound: the plane-resident kernel with 8 warps
        # per tile and tile-chained launches is the faster form there (measured 7.1 vs 9.3 us per step at 2^17 envs)
        small = per < (1 << 19) and net.n_genes <= 32
        senvs = [make_env(net, attrs, args, device, ((world * R) + rank * R + b) * args.envs, n_envs=per,
                          resident=small or None, chain=small or None) for b in range(R)]
        spool = [p[:per].contiguous() for p in pool]
        Ks = max(G, (K // 4) // G * G)
        sms = max_over_ranks(time_steps(senvs, spool, Ks, G, Wm, stream, world), device, world)
        sval = per * world * Ks / (sms * 1e-3)
        strong = {"value": sval, "unit": UNIT, "ms_per_step": sms / Ks, "steps": Ks, "envs_per_gpu": per, "total_envs": per * world,
                  "efficiency": sval / value, "efficiency_basis": "this value / the weak-scaling `value` of the same run (N x 2^20 envs)",
                  "kernel_variant": ("plane-resident state, 4 warps per 1024-env tile, tile-chained launches (PBN_STEP_CHAIN)" if small
                                     else "same kernel and launch form as the weak-scaling line")}
        for e in senvs:
            e.close()
        del senvs

    # DRAM traffic of the step kernel per launch, from the committed ncu capture of this command
    traffic = None
    tfile = ROOT / "profiles" / "traffic.json"
    if tfile.exists():
        try:
            traffic = json.loads(tfile.read_text()).get(args.net, {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None

    # end-to-end through the public API with host buffers (rank-local, every rank does it)
    import numpy as np
    e2e_env = envs[0] if not (args.resident or args.chain) else make_env(net, attrs, args, device, (2 * world * R + rank) * args.envs, resident=False, chain=False)
    host_actions = []
    for p in pool[:4]:  # the step's inputs live in pinned host memory, as the contract asks
        pa = e2e_env.pinned_actions()
        pa.copy_(p)
        host_actions.append(pa)
    n_e2e = args.e2e_steps

    packed_ok = net.n_genes <= 30
    host_actions16 = []
    if packed_ok:
        for p in pool[:4]:
            pa = e2e_env.pinned_actions16()
            pa.numpy().view(np.uint16)[...] = e2e_env.pack_actions16(p.cpu().numpy())
            host_actions16.append(pa)

    def time_e2e(compact):
        def one(i):
            if compact == "packed":
                return e2e_env.step_host(None, compact="packed", actions16=host_actions16[i % 4])
            return e2e_env.step_host(host_actions[i % 4], compact=compact)
        for i in range(12):   # warm-up: each of the 4 host buffers is seen three times (eager call, graph capture, replay)
            one(i)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ee0.record()
        for i in range(n_e2e):
            out = one(i)
        ee1.record()
        torch.cuda.synchronize()
        secs = max(time.perf_counter() - t0, ee0.elapsed_time(ee1) * 1e-3)
        t_e2e = torch.tensor([secs], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
        assert next(iter(out.values())).shape[0] == args.envs
        return args.envs * world * n_e2e / float(t_e2e.item())

    # three forms of the same results: full width (int64 state words, fp32 reward, terminated, truncated), compact
    # (uint32 state + fp32 reward + done byte, N <= 32) and packed (one uint32 = state | flags, actions as 3 x 5 bits
    # in a uint16, N <= 30: the reward follows from the caller's actions and the terminated bit via pbn_reward_table)
    e2e_full = time_e2e(False)
    compact_ok = net.n_genes <= 32
    e2e_compact = time_e2e(True) if compact_ok else None
    e2e_packed = time_e2e("packed") if packed_ok else None
    if packed_ok:
        e2e_value, (h2d, d2h) = e2e_packed, e2e_env.host_bytes_per_step_packed
        results = "one uint32 per env = state | terminated << 30 | truncated << 31; actions packed 3 x 5 bits in a uint16 (step_host(actions16=, compact='packed'))"
    elif compact_ok:
        e2e_value, (h2d, d2h) = e2e_compact, e2e_env.host_bytes_per_step_compact
        results = "uint32 state + fp32 reward + done byte per env (step_host(compact=True))"
    else:
        e2e_value, (h2d, d2h) = e2e_full, e2e_env.host_bytes_per_step
        results = "int64 state words + fp32 reward + terminated + truncated per env"
    e2e_note = {
        "results": results,
        "full_width_value": e2e_full, "full_width_d2h_bytes_per_step": e2e_env.host_bytes_per_step[1],
        "compact_value": e2e_compact, "compact_d2h_bytes_per_step": e2e_env.host_bytes_per_step_compact[1] if compact_ok else None,
        "transfer": "pbn_step_host: actions uploaded from pinned memory by the copy engine, results written "
                    "by an export kernel straight into pinned host memory (zero-copy over PCIe); packed form: 4 lanes "
                    "(upload -> unpack -> step -> export per quarter of the batch), the whole step replayed as one CUDA graph (captured per host buffer during the warm-up calls)",
        "numa": numa,
    }
    os.sched_setaffinity(0, affinity0)   # the CPU legs below use every host core again

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        arm = CpuArm(args.net, cores)
        n, busy = arm.run(seconds=args.cpu_seconds)
        arm.close()
        cpu = {"value": n / busy, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "%d processes x %.0f s of single-env oracle steps (%d env-steps), %s" % (cores, args.cpu_seconds, n, args.net)}

    extra_configs = None
    if rank == 0 and world == 1 and not args.no_configs:
        for e in envs:
            e.close()
        del envs, pool
        torch.cuda.empty_cache()
        extra_configs = run_extra_configs(args, device, stream, peak)

    if rank == 0:
        stats = dict(zip(("steps", "episodes", "terminated", "truncated", "ep_len_sum", "flips", "perturbed"),
                         stats_total.cpu().tolist()))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic", "config": workload_config(args, world, kernel),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "bytes_per_env_step": bytes_per,
                         "kernel_us": ms_per_step * 1e3},
            "cpu_baseline": cpu,
            "e2e": dict({"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                         "steps": n_e2e}, **e2e_note),
            "strong": strong,
            "configs": extra_configs,
            "gpu_launches": K,
            "clocks": clocks,
            "episode_stats": stats,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_extra_configs(args, device, stream, peak):
    """The other BASELINE.json configs, each a short run of the same protocol (rank 0, one GPU): config 2 (Bittner-10 x
    4096 envs: fixture K4 recomputed on the GPU + throughput), config 4 (70-gene network, two-word states, 2^20 envs,
    with its own roofline line), uncontrolled multi-step rollouts (pbn_rollout), and the plane-resident forms of the
    headline workload."""
    import copy
    import hashlib

    import numpy as np
    import torch
    from pbn_rl_b200 import VecPBNEnv
    out = {}
    G = 64

    def short_run(a, net, attrs, K, R, resident=False, chain=False):
        envs = [make_env(net, attrs, a, device, (100 + b) * a.envs, resident=resident, chain=chain) for b in range(R)]
        g = torch.Generator(device=device).manual_seed(77)
        pool = [torch.randint(0, net.n_genes + 1, (a.envs, 3), generator=g, device=device, dtype=torch.uint8) for _ in range(8)]
        ms = time_steps(envs, pool, K, min(G, K), 16, stream, 1)
        for e in envs:
            e.close()
        return ms / K

    # ---- config 2: Bittner-10 x 4096 envs
    net10, attrs10 = load_workload("pbn10")
    n = net10.n_genes
    x = np.array([((j + 1) * 0x9E3779B97F4A7C15) & ((1 << n) - 1) for j in range(4096)], dtype=np.uint64).reshape(-1, 1)
    jj, ii = np.arange(4096)[:, None], np.arange(n)[None, :]
    sels = [np.full((4096, n), k, dtype=np.uint8) for k in range(3)] + [((ii + jj) % 3).astype(np.uint8)]
    env = VecPBNEnv(net10, 4096, None, device=device, perturb_mode="none", horizon=0, kernel=args.kernel)
    h = hashlib.sha256()
    for sel in sels:
        env.set_state(torch.from_numpy(x.astype(np.int64)), packed=True)
        env.step_injected(None, torch.from_numpy(sel))
        torch.cuda.synchronize()
        h.update(env.state.cpu().numpy().astype("<u8").tobytes())
    env.close()
    want = json.loads((GOLD / "k4_transitions.json").read_text())["pbn10"]["sha256"]
    a10 = copy.copy(args)
    a10.net, a10.envs = "pbn10", 4096
    us = short_run(a10, net10, attrs10, 1280, 8) * 1e3
    out["pbn10_4096"] = {"value": 4096 / us * 1e6, "unit": UNIT, "us_per_step": us, "k4_known_answer_bit_exact": h.hexdigest() == want,
                         "note": "4 tiles of 1024 envs: launch-latency bound; the K4 fixture (tests/golden/k4_transitions.json) is "
                                 "recomputed with injected selections on this GPU"}
    # ---- config 4: 70-gene network, 2^20 envs, two-word states (49 algorithmic bytes per env-step)
    net70, attrs70 = load_workload("pbn70")
    a70 = copy.copy(args)
    a70.net, a70.envs = "pbn70", 1 << 20
    us_rows = short_run(a70, net70, attrs70, 640, 8) * 1e3
    us = short_run(a70, net70, attrs70, 640, 8, resident=True) * 1e3    # plane-resident state: the faster form for N > 32
    ach = BYTES_PER_STEP[2] * a70.envs / us / 1e3
    traffic = None
    try:
        traffic = json.loads((ROOT / "profiles" / "traffic.json").read_text()).get("pbn70", {}).get("dram_bytes_per_launch")
    except Exception:
        pass
    out["pbn70_2e20"] = {"value": a70.envs / us * 1e6, "unit": UNIT, "us_per_step": us, "us_per_step_row_format": us_rows,
                         "state_layout": "plane-resident (pbn_step with args->resident), 8 warps per tile",
                         "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                      "traffic": traffic, "bytes_per_env_step": BYTES_PER_STEP[2]}}
    # ---- uncontrolled rollouts: 64 updates per launch, states on chip in between (pbn_rollout)
    net28, attrs28 = load_workload("pbn28")
    a28 = copy.copy(args)
    a28.net, a28.envs = "pbn28", 1 << 20
    envs = [VecPBNEnv(net28, 1 << 20, attrs28, device=device, env_offset=(200 + b) << 20, kernel=args.kernel, **ENV_KW) for b in range(8)]
    for e in envs:
        e.rollout(4)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        for i in range(16):
            envs[i % 8].rollout(64)
        e1.record(stream)
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (16 * 64)
    for e in envs:
        e.close()
    out["rollout_pbn28"] = {"value": (1 << 20) / us * 1e6, "unit": UNIT, "us_per_update": us,
                            "note": "pbn_rollout: 64 uncontrolled updates per launch (env.step([]) x 64), p = 1e-3"}
    # ---- target membership through the hash set: the headline workload with a 15th attractor of 8192 states
    from pbn_rl_b200 import AttractorSet
    rng = np.random.default_rng(8192)
    big = {tuple(int(v) for v in rng.integers(0, 2, size=28)) for _ in range(8300)}
    attrs_big = AttractorSet(list(attrs28.attractors) + [sorted(big)[:8192]], 28)
    us_h = short_run(a28, net28, attrs_big, 640, 8) * 1e3
    out["membership_hashset_pbn28"] = {"us_per_step": us_h, "value": (1 << 20) / us_h * 1e6, "unit": UNIT, "attractors": 15, "largest_attractor": 8192,
                                       "note": "targets uniform over 14 single-state attractors + one 8192-state attractor: single-state targets are "
                                               "compared in shared memory, the envs of the large target probe the L2-resident hash set over "
                                               "its 8192 states (pbn_update_attractors)"}
    # ---- real selection probabilities (what ASSA-format PBNs carry): the headline network with weights 0.5 / 0.3 / 0.2 on
    # every gene's three predictors -- bit-sliced threshold comparison instead of the pair-plane draw
    from pbn_rl_b200 import PBNNetwork
    net_w = PBNNetwork(list(net28.genes), [list(fs) for fs in net28.functions],
                       [[0.5, 0.3, 0.2][:len(fs)] if len(fs) == 3 else [1.0 / len(fs)] * len(fs) for fs in net28.functions], "pbn28_weighted")
    us_w = short_run(a28, net_w, attrs28, 640, 8) * 1e3
    out["weighted_pbn28"] = {"us_per_step": us_w, "value": (1 << 20) / us_w * 1e6, "unit": UNIT,
                             "note": "Bittner-28 with selection probabilities 0.5 / 0.3 / 0.2 per gene (train_assa_matlab_BQN.py:72-171 style): "
                                     "bit-sliced kernel, predictor index = number of 32-bit thresholds <= a bit-sliced 32-bit uniform"}
    # ---- the headline workload with plane-resident env state (same random streams, bit-identical results)
    if not (args.resident or args.chain):
        try:
            us_r = short_run(a28, net28, attrs28, 640, 8, resident=True) * 1e3
            us_c = short_run(a28, net28, attrs28, 640, 8, resident=True, chain=True) * 1e3
            out["resident_pbn28"] = {"us_per_step_pdl": us_r, "us_per_step_chained": us_c,
                                     "note": "pbn_step with args->resident (csrc/step_planes.cuh): no transposes and 29 instead of 33 "
                                             "bytes per env-step, but the auto-reset scatter into the planes makes it slower than the "
                                             "row-format kernel on this workload (5 % of the envs reset per step)"}
        except Exception as exc:   # the resident form is optional
            out["resident_pbn28"] = {"error": str(exc)[:200]}
    return out


_JSON_FD = None


def emit(line):
    """The ONE JSON line of the contract, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    # stdout carries exactly one JSON line: anything libraries print to fd 1 (NCCL's version banner, ...) is
    # sent to stderr instead
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--net", default="pbn28")
    ap.add_argument("--envs", type=int, default=1 << 20, help="env instances per GPU")
    ap.add_argument("--batches", type=int, default=8, help="independent env batches rotated to defeat L2")
    ap.add_argument("--action-pool", type=int, default=16)
    ap.add_argument("--graph-steps", type=int, default=64)
    ap.add_argument("--kernel", default="auto")
    ap.add_argument("--e2e-steps", type=int, default=30)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pdl", action="store_true", help="plain stream-serialised launches instead of programmatic dependent launch")
    ap.add_argument("--resident", action="store_true", help="plane-resident env state (pbn_step with args->resident)")
    ap.add_argument("--chain", action="store_true", help="plane-resident state with tile-chained launches (PBN_STEP_CHAIN)")
    ap.add_argument("--strong", action="store_true", help="also time the strong-scaling form at N = 1 (envs / N per GPU)")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configs (pbn10 x 4096, pbn70, rollout)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step (rank 0) as DIR/<name>.npy; the inputs are seeded, so two "
                         "builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.impl == "reference":
        args.steps_ref = args.steps if args.steps is not None else 20
        args.warmup_ref = args.warmup if args.warmup is not None else 3
        run_reference(args)
        return
    args.steps = args.steps if args.steps is not None else 6400
    args.warmup = args.warmup if args.warmup is not None else 64
    use_private_jit_cache()
    run_gpu(args)


if __name__ == "__main__":
    main()
