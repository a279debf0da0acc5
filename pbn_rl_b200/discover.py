"""Attractor discovery and steady-state statistics on the GPU (SURVEY.md 8f-3).

What the reference does on the host: ``graph.genSTG()`` + networkx SCC condensation for small nets
(print_graph.py:15-34), an external tool (CABEAN / ASSA-PBN, SURVEY.md Appendix A) for the cached
``data/attractors_*.pkl``, attractors found *during* training for the large ones
(``env.all_attractors`` grows, bdq_model/__init__.py:182-184) and ``compute_ssd_hist`` (300 x 10^5 env
steps, train_pbn_28.py:257) for steady-state histograms.

Here:
* :func:`find_attractors_rollout` -- for any N <= 128: 2^k perturbation-free rollouts on the GPU
  (``pbn_step``), their end states counted in a device hash table (``pbn_visit_count``); every distinct
  end state is a candidate from which the host takes the *forward closure* under the STG successor
  relation (successor descriptors from ``pbn_successor_sets``).  A closed set's sink SCCs are sink SCCs of
  the whole STG, so every attractor returned is exact (closed and strongly connected); what is sampled is
  only *which* attractors are found (those with a basin the rollouts hit).
* :func:`steady_state_histogram` -- visit counts of (projected) states over many perturbed steps.
* :func:`steady_state_statistics` / :class:`StateRecorder` -- per-gene ON frequencies and the distribution of the
  state projected onto up to 12 genes, counted on the device (``pbn_rollout_record`` inside the rollout kernel,
  ``pbn_record_states`` after a step); full states of more than 12 genes go through :func:`steady_state_histogram`.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from ._cabi import check
from .attractors import AttractorSet
from .network import PBNNetwork
from .vec_env import VecPBNEnv

__all__ = ["VisitCounter", "find_attractors_rollout", "attractor_reached_from", "basin_labels", "steady_state_histogram", "successor_descriptors",
           "forward_closure", "sink_sccs_of_closed_set", "StateRecorder", "steady_state_statistics"]


def _words_to_int(words: Sequence[int]) -> int:
    v = 0
    for k, w in enumerate(words):
        v |= (int(w) & 0xFFFFFFFFFFFFFFFF) << (64 * k)
    return v


def _int_to_words(v: int, w: int) -> List[int]:
    return [(v >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(w)]


class VisitCounter:
    """Device hash table state -> visit count (``pbn_visit_count``)."""

    def __init__(self, env: VecPBNEnv, capacity: int = 1 << 20):
        if capacity < 2 or capacity & (capacity - 1):
            raise ValueError("capacity must be a power of two")
        self.env, self.capacity = env, int(capacity)
        dev = env.device
        self.tags = torch.zeros((capacity,), dtype=torch.int64, device=dev)
        self.slot_state = torch.zeros((capacity, env.n_words), dtype=torch.int64, device=dev)
        self.counts = torch.zeros((capacity,), dtype=torch.int64, device=dev)
        self.overflow = torch.zeros((1,), dtype=torch.int32, device=dev)

    def add(self, states: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None) -> None:
        env = self.env
        states = env.state if states is None else states.to(device=env.device, dtype=torch.int64).contiguous()
        if mask is not None:
            mask = mask.to(device=env.device, dtype=torch.uint8).contiguous()
        check(env.lib.pbn_visit_count(env._h, states.data_ptr(), None if mask is None else mask.data_ptr(),
                                      states.shape[0], self.tags.data_ptr(), self.slot_state.data_ptr(),
                                      self.counts.data_ptr(), self.capacity, self.overflow.data_ptr(), env._stream()))

    def items(self) -> Tuple[np.ndarray, np.ndarray]:
        """``(states [K, W] uint64, counts [K] int64)`` of the occupied slots, most visited first."""
        if int(self.overflow.item()):
            raise RuntimeError("visit-count table overflowed (%d states found no slot): raise capacity" % int(self.overflow.item()))
        used = torch.nonzero(self.tags != 0).reshape(-1)
        st = self.slot_state[used].cpu().numpy().astype(np.uint64)
        ct = self.counts[used].cpu().numpy()
        order = np.lexsort(tuple(st[:, k] for k in range(st.shape[1])) + (-ct,))
        return st[order], ct[order]


def successor_descriptors(env: VecPBNEnv, states: Sequence[int]) -> List[Tuple[int, int]]:
    """``[(can1, can0)]`` python ints per state (``pbn_successor_sets``)."""
    w = env.n_words
    arr = np.array([_int_to_words(s, w) for s in states], dtype=np.uint64).reshape(-1, w)
    d = torch.from_numpy(arr.astype(np.int64)).to(env.device)
    c1, c0 = torch.empty_like(d), torch.empty_like(d)
    check(env.lib.pbn_successor_sets(env._h, d.data_ptr(), d.shape[0], c1.data_ptr(), c0.data_ptr(), env._stream()))
    c1, c0 = c1.cpu().numpy().astype(np.uint64), c0.cpu().numpy().astype(np.uint64)
    return [(_words_to_int(c1[k]), _words_to_int(c0[k])) for k in range(len(states))]


def _expand(can1: int, can0: int, max_free: int) -> Optional[List[int]]:
    free = can1 & can0
    nfree = bin(free).count("1")
    if nfree > max_free:
        return None
    out = [can1 & ~free]
    b = free
    while b:
        low = b & -b
        out += [t | low for t in out]
        b ^= low
    return out


def forward_closure(env: VecPBNEnv, start: int, max_states: int = 1 << 16, max_free: int = 16) -> Optional[Dict[int, List[int]]]:
    """All states reachable from ``start`` in the perturbation-free STG as ``{state: successors}``, or
    ``None`` if the closure exceeds ``max_states`` (or one state has more than 2^max_free successors).
    Breadth first; each frontier's successor descriptors come from one ``pbn_successor_sets`` launch."""
    graph: Dict[int, List[int]] = {}
    frontier = [start]
    seen = {start}
    while frontier:
        desc = successor_descriptors(env, frontier)
        nxt: List[int] = []
        for s, (c1, c0) in zip(frontier, desc):
            succ = _expand(c1, c0, max_free)
            if succ is None:
                return None
            graph[s] = succ
            for t in succ:
                if t not in seen:
                    seen.add(t)
                    nxt.append(t)
        if len(seen) > max_states:
            return None
        frontier = nxt
    return graph


def sink_sccs_of_closed_set(graph: Dict[int, List[int]]) -> List[List[int]]:
    """Sink strongly-connected components of a closed sub-graph (iterative Tarjan): attractors."""
    index: Dict[int, int] = {}
    low: Dict[int, int] = {}
    comp: Dict[int, int] = {}
    on_stack = set()
    stack: List[int] = []
    counter = 0
    n_comp = 0
    for root in graph:
        if root in index:
            continue
        work = [(root, 0)]
        while work:
            v, pi = work.pop()
            if pi == 0:
                index[v] = low[v] = counter
                counter += 1
                stack.append(v)
                on_stack.add(v)
            recurse = False
            sv = graph[v]
            for k in range(pi, len(sv)):
                w = sv[k]
                if w not in index:
                    work.append((v, k + 1))
                    work.append((w, 0))
                    recurse = True
                    break
                if w in on_stack:
                    low[v] = min(low[v], index[w])
            if recurse:
                continue
            if low[v] == index[v]:
                while True:
                    w = stack.pop()
                    on_stack.discard(w)
                    comp[w] = n_comp
                    if w == v:
                        break
                n_comp += 1
            if work:
                parent = work[-1][0]
                low[parent] = min(low[parent], low[v])
    sink = [True] * n_comp
    for s, succ in graph.items():
        for t in succ:
            if comp[t] != comp[s]:
                sink[comp[s]] = False
    members: Dict[int, List[int]] = {}
    for s in graph:
        if sink[comp[s]]:
            members.setdefault(comp[s], []).append(s)
    return sorted(sorted(m) for m in members.values())


class _ClosureWorkspace:
    """Device buffers of the closure search: the state list, the hash table and the flags."""

    def __init__(self, env: VecPBNEnv, max_states: int):
        dev, w = env.device, env.n_words
        self.env, self.max_states = env, int(max_states)
        cap = 2
        while cap < 4 * self.max_states:
            cap *= 2
        self.capacity = cap
        self.list = torch.zeros((self.max_states, w), dtype=torch.int64, device=dev)
        self.tags = torch.zeros((cap,), dtype=torch.int64, device=dev)
        self.slot_state = torch.zeros((cap, w), dtype=torch.int64, device=dev)
        self.slot_index = torch.zeros((cap,), dtype=torch.int64, device=dev)
        self.flags = torch.zeros((self.max_states,), dtype=torch.uint8, device=dev)
        self.list_count = torch.zeros((1,), dtype=torch.int64, device=dev)
        self.status = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.changed = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.overflow = torch.zeros((1,), dtype=torch.int32, device=dev)


def attractor_reached_from(env: VecPBNEnv, seed_state: int, ws: Optional[_ClosureWorkspace] = None,
                           max_states: int = 1 << 16, max_free: int = 16, max_restarts: int = 64) -> Optional[List[int]]:
    """The attractor (sink SCC of the perturbation-free STG) inside the forward closure of ``seed_state``,
    computed on the device: breadth-first closure (``pbn_closure_expand``: one CTA per frontier state
    enumerates its 2^free successors into a hash set), then backward reachability to the seed
    (``pbn_closure_reach``).  If every closure state reaches the seed, the closure is the attractor;
    otherwise the search restarts from a state that does not (its closure is strictly smaller).
    Returns the sorted member states, or ``None`` if a closure exceeds ``max_states`` / ``max_free``."""
    ws = ws or _ClosureWorkspace(env, max_states)
    lib, h, w = env.lib, env._h, env.n_words
    cand = seed_state
    for _ in range(max_restarts):
        ws.tags.zero_()
        ws.slot_index.zero_()
        ws.status.zero_()
        ws.list[0] = torch.tensor([x - (1 << 64) if x >= (1 << 63) else x for x in _int_to_words(cand, w)], dtype=torch.int64)
        ws.list_count.fill_(1)
        check(lib.pbn_visit_count(h, ws.list.data_ptr(), None, 1, ws.tags.data_ptr(), ws.slot_state.data_ptr(),
                                  ws.slot_index.data_ptr(), ws.capacity, ws.overflow.data_ptr(), env._stream()))
        begin, end = 0, 1
        while begin < end:
            check(lib.pbn_closure_expand(h, ws.list.data_ptr(), begin, end, ws.max_states, ws.list_count.data_ptr(),
                                         ws.tags.data_ptr(), ws.slot_state.data_ptr(), ws.slot_index.data_ptr(),
                                         ws.capacity, int(max_free), ws.status.data_ptr(), env._stream()))
            if int(ws.status.item()) != 0:
                return None
            begin, end = end, int(ws.list_count.item())
        count = end
        ws.flags[:count] = 0
        ws.flags[0] = 1
        while True:
            ws.changed.zero_()
            check(lib.pbn_closure_reach(h, ws.list.data_ptr(), count, ws.flags.data_ptr(), ws.tags.data_ptr(),
                                        ws.slot_state.data_ptr(), ws.slot_index.data_ptr(), ws.capacity, ws.changed.data_ptr(), env._stream()))
            if int(ws.changed.item()) == 0:
                break
        flags = ws.flags[:count]
        members = ws.list[:count].cpu().numpy().astype(np.uint64)
        if bool(flags.all().item()):
            return sorted(_words_to_int(members[k]) for k in range(count))
        first = int(torch.nonzero(flags == 0)[0].item())
        cand = _words_to_int(members[first])
    return None


def find_attractors_rollout(network: PBNNetwork, n_rollouts: int = 1 << 16, burn_in: int = 256,
                            device: Union[str, torch.device] = "cuda:0", seed: int = 0x5EED,
                            max_attractor_states: int = 1 << 14, max_candidates: int = 4096,
                            table_capacity: int = 1 << 20, kernel: str = "auto", method: str = "device",
                            max_unresolved: int = 8):
    """Attractors (sink SCCs of the perturbation-free STG) reachable from ``n_rollouts`` uniformly random
    initial states.  Returns ``(AttractorSet, info)``; attractors are sorted by smallest state like
    :func:`find_attractors_stg`, ``info['basin_fraction']`` estimates the share of the state space draining
    into each one, ``info['unresolved']`` lists candidates whose closure exceeded ``max_attractor_states``.
    ``method="device"`` runs closure + connectivity on the GPU (:func:`attractor_reached_from`),
    ``method="host"`` the python closure + Tarjan (small networks, cross-check).  Candidates are tried
    from the most visited end state down; the search stops after ``max_unresolved`` failures."""
    n, w = network.n_genes, network.n_words
    e = ((int(n_rollouts) + 1023) // 1024) * 1024
    env = VecPBNEnv(network, e, None, device=device, seed=seed, horizon=0, bins=1, perturb_p=0.0, kernel=kernel)
    dev = env.device
    g = torch.Generator(device=dev).manual_seed(int(seed) & 0x7FFFFFFF)
    for k in range(w):
        bits = min(64, n - 64 * k)
        hi = torch.randint(0, 1 << max(bits - 31, 0), (e,), generator=g, device=dev, dtype=torch.int64)
        lo = torch.randint(0, 1 << min(bits, 31), (e,), generator=g, device=dev, dtype=torch.int64)
        env.state[:, k] = (hi << 31) | lo
    env.rollout(int(burn_in), stats=False)       # one launch: the states stay on chip between the updates
    table = VisitCounter(env, table_capacity)
    table.add()
    states, counts = table.items()
    order = np.argsort(-counts, kind="stable")
    owner: Dict[int, int] = {}          # state -> attractor index
    attractors: List[List[int]] = []
    hits: List[int] = []
    unresolved: List[int] = []
    ws = _ClosureWorkspace(env, max_attractor_states) if method == "device" else None
    for k in order[:max_candidates]:
        s = _words_to_int(states[k])
        if s in owner:
            hits[owner[s]] += int(counts[k])
            continue
        if method == "device":
            found = attractor_reached_from(env, s, ws, max_states=max_attractor_states)
            sccs = None if found is None else [found]
        else:
            closure = forward_closure(env, s, max_states=max_attractor_states)
            sccs = None if closure is None else sink_sccs_of_closed_set(closure)
        if sccs is None:
            unresolved.append(s)
            if len(unresolved) >= max_unresolved:
                break       # the rarely-visited tail: transient end states with huge closures (burn-in too short)
            continue
        for scc in sccs:
            if scc[0] in owner:
                continue
            idx = len(attractors)
            attractors.append(scc)
            hits.append(0)
            for t in scc:
                owner[t] = idx
        if s in owner:      # transient end states (burn-in too short) are not credited to any attractor
            hits[owner[s]] += int(counts[k])
    env.close()
    perm = sorted(range(len(attractors)), key=lambda i: attractors[i][0])
    attrs = [[tuple((s >> i) & 1 for i in range(n)) for s in attractors[i]] for i in perm]
    info = {"n_rollouts": e, "burn_in": int(burn_in), "distinct_end_states": int(len(counts)),
            "basin_fraction": [hits[i] / e for i in perm], "unresolved": unresolved,
            "states": [attractors[i] for i in perm]}
    return AttractorSet(attrs, n), info


def basin_labels(env: VecPBNEnv, max_steps: int = 1024, chunk: int = 8) -> Tuple[torch.Tensor, torch.Tensor]:
    """Which attractor every instance drains into when left alone: the loop of the basin classifier
    (graph_classifier/__init__.py:125-148 rolls ``env.step([])`` until ``env.is_attracting_state(state)``), for all
    instances at once.  Rolls ``chunk`` uncontrolled updates at a time (``pbn_rollout``) until every state lies in
    an attractor of the env's table or ``max_steps`` is reached.  Returns ``(attractor_id [E] int32, -1 = none
    reached, steps_taken [E] int32 rounded up to a multiple of ``chunk``)``; the env's states are left where the
    rollouts ended."""
    ids = env.attractor_ids()
    steps = torch.zeros((env.num_envs,), dtype=torch.int32, device=env.device)
    done = 0
    while done < max_steps and bool((ids < 0).any().item()):
        n = min(chunk, max_steps - done)
        env.rollout(n, stats=False)
        done += n
        new = env.attractor_ids()
        steps = torch.where((ids < 0) & (new >= 0), torch.full_like(steps, done), steps)
        ids = torch.where(ids < 0, new, ids)     # the first attractor reached (attractors are closed when p = 0)
    return ids, steps


def steady_state_histogram(env: VecPBNEnv, steps: int, actions: Optional[torch.Tensor] = None,
                           genes: Optional[Sequence[int]] = None, burn_in: int = 0,
                           table_capacity: int = 1 << 22) -> Dict[int, int]:
    """Visit counts of the states (restricted to ``genes``, packed in that order, if given) seen by all
    instances of ``env`` over ``steps`` steps after ``burn_in`` steps -- the histogram behind
    ``compute_ssd_hist`` (train_pbn_28.py:257).  ``{state int: visits}``; sums to ``steps * num_envs``."""
    if actions is None and env.step_ctr_dev is None:
        env.rollout(int(burn_in), stats=False)
    else:
        for _ in range(int(burn_in)):
            env.step(actions, stats=False)
    table = VisitCounter(env, table_capacity)
    proj = None
    if genes is not None:
        genes = list(genes)
        if len(genes) > 63:
            raise ValueError("at most 63 genes in a projection")
        proj = torch.zeros((env.num_envs, env.n_words), dtype=torch.int64, device=env.device)
    for _ in range(int(steps)):
        env.step(actions, stats=False)
        if proj is None:
            table.add()
        else:
            proj.zero_()
            for j, gi in enumerate(genes):
                proj[:, 0] |= ((env.state[:, gi >> 6] >> (gi & 63)) & 1) << j
            table.add(proj)
    states, counts = table.items()
    return {_words_to_int(states[k]): int(counts[k]) for k in range(len(counts))}


class StateRecorder:
    """Device accumulators of steady-state statistics for the states of ``env``: per-gene ON counts
    (``marginals=True``) and the histogram of the states projected onto ``genes`` (at most 12 distinct genes; bin
    bit j = gene ``genes[j]``, the packing of :func:`steady_state_histogram`; ``genes=None`` keeps no histogram,
    ``genes=[]`` one bin counting every state).  Counts only ever grow: :meth:`add` and
    ``env.rollout(n, recorder=...)`` add to them."""

    def __init__(self, env: VecPBNEnv, genes: Optional[Sequence[int]] = None, marginals: bool = True):
        self.env = env
        self.genes = None if genes is None else [int(g) for g in genes]
        if self.genes is not None:
            if len(self.genes) > 12:
                raise ValueError("at most 12 genes in a projection (full states: steady_state_histogram)")
            if len(set(self.genes)) != len(self.genes) or any(g < 0 or g >= env.n_genes for g in self.genes):
                raise ValueError("projection genes must be distinct and in [0, %d)" % env.n_genes)
        self.k = 0 if self.genes is None else len(self.genes)
        self._proj = (C.c_int32 * 12)(*(self.genes or []))
        self._proj_ptr = C.addressof(self._proj)
        dev = env.device
        self.gene_on = torch.zeros((env.n_genes,), dtype=torch.int64, device=dev) if marginals else None
        self.hist = torch.zeros((1 << self.k,), dtype=torch.int64, device=dev) if self.genes is not None else None
        self.n = 0   # recorded env-states

    def add(self, states: Optional[torch.Tensor] = None) -> None:
        """Record ``states`` (row-format ``[E, W]`` words; default: the env's current states) once."""
        env = self.env
        states = env.state if states is None else states.to(device=env.device, dtype=torch.int64).contiguous()
        if states.dim() != 2 or states.shape[1] != env.n_words:
            raise ValueError("states must be [E, %d] int64 words" % env.n_words)
        check(env.lib.pbn_record_states(env._h, states.data_ptr(), states.shape[0], self._proj_ptr, self.k,
                                        None if self.gene_on is None else self.gene_on.data_ptr(),
                                        None if self.hist is None else self.hist.data_ptr(), env._stream()))
        self.n += int(states.shape[0])

    def counts(self) -> Tuple[Optional[np.ndarray], Optional[np.ndarray]]:
        """The raw accumulators ``(gene_on [N], hist [2^k])`` as uint64 arrays (``None`` where not kept)."""
        f = (lambda t: None if t is None else t.cpu().numpy().astype(np.uint64))
        return f(self.gene_on), f(self.hist)

    def marginals(self) -> np.ndarray:
        """P(gene g is ON) over the recorded states, float64 ``[N]``."""
        if self.gene_on is None:
            raise ValueError("this recorder keeps no per-gene counts (marginals=False)")
        return self.gene_on.cpu().numpy().astype(np.float64) / max(self.n, 1)

    def distribution(self) -> np.ndarray:
        """Frequency of every projected state over the recorded states, float64 ``[2^k]``."""
        if self.hist is None:
            raise ValueError("this recorder keeps no histogram (genes=None)")
        return self.hist.cpu().numpy().astype(np.float64) / max(self.n, 1)


def steady_state_statistics(env: VecPBNEnv, steps: int, burn_in: int = 0, genes: Optional[Sequence[int]] = None,
                            stride: int = 1, policy: Optional[Callable[[torch.Tensor], torch.Tensor]] = None,
                            marginals: bool = True) -> StateRecorder:
    """Steady-state statistics of ``env``'s network (``compute_ssd_hist``, train_pbn_28.py:257): ``burn_in`` steps,
    then ``steps`` more, recording every instance's state after each step ``s`` (``s = 1..steps``) with
    ``s % stride == 0``.  Returns the :class:`StateRecorder` (``marginals()``, ``distribution()`` over ``genes``).

    Without ``policy`` the network runs uncontrolled: ``env.rollout(burn_in)`` and ``env.rollout(steps,
    recorder=..., stride=stride)``, the recording fused into the rollout kernel on the sliced kernel.  With
    ``policy(obs) -> actions`` the agent acts at every step: ``observe -> policy -> step -> record``, the
    controlled steady state ``compute_ssd_hist(env, model)`` estimates.  Actions are uint8 ``[E, bins]`` as
    :meth:`VecPBNEnv.step` takes them; the env's horizon, targets and auto-reset apply as in any other step."""
    rec = StateRecorder(env, genes=genes, marginals=marginals)
    if policy is None:
        env.rollout(int(burn_in), stats=False)
        env.rollout(int(steps), stats=False, recorder=rec, stride=int(stride))
        return rec
    if int(stride) < 1:
        raise ValueError("stride must be >= 1")
    for s in range(1, int(burn_in) + int(steps) + 1):
        env.step(policy(env.observe()), stats=False)
        if s > int(burn_in) and (s - int(burn_in)) % int(stride) == 0:
            rec.add()
    return rec
