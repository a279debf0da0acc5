"""TEST INFRASTRUCTURE -- CPU restatement ("oracle") of the PBN environment hot path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product (pbn_rl_b200) never does.

What is restated, and from where
--------------------------------
The arithmetic of the path lives in a third-party dependency that is NOT in /root/reference:
``gym-PBN[vis]==1.1.1`` (reference: requirements.txt:11; a private fork -- the env ids and
methods the scripts use do not exist upstream, SURVEY.md section 0).  It cannot be installed
here (no network).  This file therefore restates the *published* PBN semantics
(Shmulevich et al. 2002: synchronous update, per-gene random predictor selection, random
gene perturbation) and anchors every API detail on the reference's own call sites:

* action encoding, 0 = no-op, k>=1 flips gene k-1, set semantics   bdq_model/__init__.py:76-84,176-177
* reset()/step() tuple shapes, done = terminated | truncated          bdq_model/__init__.py:161,177,186,204
* setState / setTarget / in_target / render, '*' -> 0                 model_tester.py:595-625
* step([]) = one uncontrolled network update                          graph_classifier/__init__.py:121-148
* int action, n_steps                                                 ddqn_per/__init__.py:341-354
* ISPL -> python boolean expression strings evaluated per gene        train_assa_BQN.py:51-109
* uniform 1/k predictor selection                                     train_pbn_28.py:139-151

Parity pins (tests/test_oracle_golden.py): the deterministic Boolean update is pinned by the
data-file known answers K2/K4/K5 derived from the reference tree (kaban/*.ispl,
data/attractors_Bittner-7.pkl; SURVEY.md section 8c) -- fixtures in tests/golden/.  The
reference's own tests hold NOTHING for this path (SURVEY.md section 4), and the fork's
perturbation model, perturbation rate and reward constants are not evidenced anywhere in
the tree: for those the parity is UNPINNED ("parity unpinned"); they are explicit
parameters here and in the product, and the bit-exact contract is defined on the
deterministic core T(state, flip_mask, sel, pert_mask).

Like gym-PBN, the per-instance env below evaluates each predictor with python ``eval`` on a
name->bool dict and draws randomness from python ``random`` -- that is the point: it is the
CPU baseline that gets timed next to the GPU path.
"""
from __future__ import annotations

import json
import random
import re
from pathlib import Path
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from .philox_ref import philox4x32

PERT_NONE, PERT_A, PERT_B, PERT_C = 0, 1, 2, 3
PERT_MODES = {"none": 0, "A": 1, "B": 2, "C": 3, 0: 0, 1: 1, 2: 2, 3: 3}

# Philox counter layout shared with the kernels (include/pbn_b200.h, "Random streams")
KIND_SELECT, KIND_PERTURB, KIND_RESET = 0, 1, 2


# --------------------------------------------------------------------------------------
# network
# --------------------------------------------------------------------------------------

def _to_python_expr(expr: str) -> str:
    e = re.sub(r"([A-Za-z_]\w*)\s*=\s*false", r"( not \1 )", expr)
    e = re.sub(r"([A-Za-z_]\w*)\s*=\s*true", r"\1", e)
    e = e.replace("||", "|").replace("&&", "&").replace("!", "~")
    e = e.replace("~", " not ").replace("&", " and ").replace("|", " or ")
    e = re.sub(r"\btrue\b", "True", e)
    e = re.sub(r"\bfalse\b", "False", e)
    return e.strip()


def _to_numpy_expr(py_expr: str) -> str:
    e = re.sub(r"\bnot\b", "~", py_expr)
    e = re.sub(r"\band\b", "&", e)
    e = re.sub(r"\bor\b", "|", e)
    return e.strip()


def read_ispl(text: str) -> Tuple[List[str], Dict[str, List[str]]]:
    """Independent minimal ISPL reader (both dialects of SURVEY.md Appendix A)."""
    genes: List[str] = []
    funcs: Dict[str, List[str]] = {}
    section = None
    for raw in text.splitlines():
        line = raw.strip()
        if not line:
            continue
        if line.startswith("Vars:"):
            section = "vars"
        elif line.startswith("Evolution:"):
            section = "evo"
        elif line.startswith("end"):
            section = None
        elif section == "vars":
            name = line.split(":")[0].strip()
            genes.append(name)
            funcs[name] = []
        elif section == "evo":
            m = re.match(r"^(\w+)\s*=\s*(true|false)\s+if\s+(.*)=\s*(true|false)\s*;?$", line)
            assert m, line
            if m.group(2) == "true":
                assert m.group(4) == "true", line
                funcs[m.group(1)].append(m.group(3).strip())
    return genes, funcs


class OracleNetwork:
    """Genes + predictor expressions, evaluated with ``eval`` (python or numpy namespace)."""

    def __init__(self, genes: Sequence[str], exprs: Sequence[Sequence], name: str = ""):
        self.genes = list(genes)
        self.n = len(self.genes)
        self.name = name
        self.exprs: List[List[str]] = []
        self.probs: List[List[float]] = []
        for row in exprs:
            es, ps = [], []
            for item in row:
                if isinstance(item, (tuple, list)):
                    es.append(str(item[0]))
                    ps.append(float(item[1]))
                else:
                    es.append(str(item))
                    ps.append(None)
            if any(p is None for p in ps):
                ps = [1.0 / len(es)] * len(es)
            tot = sum(ps)
            self.exprs.append(es)
            self.probs.append([p / tot for p in ps])
        self.py_src = [[_to_python_expr(e) for e in es] for es in self.exprs]
        self.py_code = [[compile(s, "<pbn>", "eval") for s in row] for row in self.py_src]
        self.np_code = [[compile(_to_numpy_expr(s), "<pbn-np>", "eval") for s in row] for row in self.py_src]
        self.words = 1 if self.n <= 64 else 2

    @classmethod
    def from_ispl(cls, text: str, name: str = "") -> "OracleNetwork":
        genes, funcs = read_ispl(text)
        return cls(genes, [funcs[g] for g in genes], name)

    @classmethod
    def from_json(cls, path) -> "OracleNetwork":
        d = json.loads(Path(path).read_text())
        return cls(d["genes"], d["functions"], d.get("name", ""))

    # --- deterministic core T (SURVEY.md 8a-4), one instance, python ints as bit sets
    def transition(self, state: int, flip_mask: int, sel: Sequence[int], pert_mask: int, mode=PERT_A) -> int:
        mode = PERT_MODES[mode]
        s1 = state ^ flip_mask
        env = {g: bool((s1 >> i) & 1) for i, g in enumerate(self.genes)}
        f = 0
        for i in range(self.n):
            if eval(self.py_code[i][sel[i]], {}, env):
                f |= 1 << i
        if mode == PERT_NONE:
            return f
        if mode == PERT_A:
            return (s1 ^ pert_mask) if pert_mask else f
        if mode == PERT_B:
            return f ^ pert_mask
        full = (1 << self.n) - 1
        return (f & ~pert_mask & full) | (~s1 & pert_mask & full)

    # --- the same, vectorised over E instances with numpy (for large-E parity checks)
    def transition_batch(self, words: np.ndarray, flip_words: np.ndarray, sel: np.ndarray,
                         pert_words: np.ndarray, mode=PERT_A) -> np.ndarray:
        mode = PERT_MODES[mode]
        words = np.asarray(words, dtype=np.uint64).reshape(-1, self.words)
        s1 = words ^ np.asarray(flip_words, dtype=np.uint64).reshape(-1, self.words)
        pert = np.asarray(pert_words, dtype=np.uint64).reshape(-1, self.words)
        sel = np.asarray(sel).reshape(-1, self.n)
        ns = {g: ((s1[:, i >> 6] >> np.uint64(i & 63)) & np.uint64(1)).astype(bool)
              for i, g in enumerate(self.genes)}
        e = s1.shape[0]
        f = np.zeros_like(s1)
        for i in range(self.n):
            vals = np.zeros(e, dtype=bool)
            for k in range(len(self.np_code[i])):
                v = eval(self.np_code[i][k], {}, ns)
                v = np.broadcast_to(np.asarray(v, dtype=bool), (e,))
                vals = np.where(sel[:, i] == k, v, vals)
            f[:, i >> 6] |= vals.astype(np.uint64) << np.uint64(i & 63)
        if mode == PERT_NONE:
            return f
        if mode == PERT_A:
            any_p = (pert != 0).any(axis=1, keepdims=True)
            return np.where(any_p, s1 ^ pert, f)
        if mode == PERT_B:
            return f ^ pert
        return (f & ~pert) | (~s1 & pert & self.mask_words())

    def mask_words(self) -> np.ndarray:
        n = self.n
        if n <= 64:
            return np.array([(1 << n) - 1], dtype=np.uint64)
        return np.array([(1 << 64) - 1, (1 << (n - 64)) - 1], dtype=np.uint64)


# --------------------------------------------------------------------------------------
# attractor helpers (reference format: list[list[tuple(0/1/'*')]])
# --------------------------------------------------------------------------------------

def state_matches(pattern: Sequence, state: Sequence[int]) -> bool:
    return all(p == "*" or int(p) == int(x) for p, x in zip(pattern, state))


def attractor_contains(attractor: Sequence[Sequence], state: Sequence[int]) -> bool:
    return any(state_matches(p, state) for p in attractor)


def attractor_tables(attractors, n: int):
    """(offset, care[S,W], val[S,W]) -- independent restatement of the device table layout."""
    w = 1 if n <= 64 else 2
    offs, care, val = [0], [], []
    for attr in attractors:
        for s in attr:
            c, v = [0] * w, [0] * w
            for i, b in enumerate(s):
                if b == "*":
                    continue
                c[i >> 6] |= 1 << (i & 63)
                if int(b):
                    v[i >> 6] |= 1 << (i & 63)
            care.append(c)
            val.append(v)
        offs.append(len(care))
    return (np.array(offs, dtype=np.int32), np.array(care, dtype=np.uint64).reshape(-1, w),
            np.array(val, dtype=np.uint64).reshape(-1, w))


def bits_to_int(bits: Sequence[int]) -> int:
    v = 0
    for i, b in enumerate(bits):
        if b != "*" and int(b):
            v |= 1 << i
    return v


def int_to_bits(v: int, n: int) -> Tuple[int, ...]:
    return tuple((v >> i) & 1 for i in range(n))


# --------------------------------------------------------------------------------------
# step semantics shared by the per-instance env and the batched restatement
# --------------------------------------------------------------------------------------

def flip_mask_from_actions(actions: Sequence[int], n: int) -> int:
    """Set semantics: duplicates do not cancel (SURVEY.md Appendix B); 0 and values > n are no-ops."""
    m = 0
    for a in actions:
        a = int(a)
        if 1 <= a <= n:
            m |= 1 << (a - 1)
    return m


def reward_f32(n_flips: int, hit: bool, r_success: float, r_step: float, r_action: float, wrong: bool = False,
               r_wrong: float = 0.0) -> np.float32:
    """reward = (r_step + r_action * n_flips) + (r_success if hit else r_wrong if wrong else 0), each op rounded to
    fp32.  `wrong`: the step ended in an attractor that is not the target (upstream gym-PBN's penalty, SURVEY.md 8c)."""
    base = np.float32(r_step) + np.float32(r_action) * np.float32(n_flips)
    bonus = np.float32(r_success) if hit else (np.float32(r_wrong) if wrong else np.float32(0.0))
    return np.float32(base + bonus)


class OraclePBNEnv:
    """Per-instance gym-style PBN env (the CPU baseline).  One python object = one env."""

    def __init__(self, network: OracleNetwork, attractors, horizon: int = 20, perturb_p: float = 0.0,
                 perturb_mode="A", r_success: float = 5.0, r_step: float = 0.0, r_action: float = -1.0,
                 seed: Optional[int] = None, r_wrong: float = 0.0):
        self.net = network
        self.n = network.n
        self.all_attractors = [list(map(tuple, a)) for a in attractors]
        self.horizon = int(horizon)
        self.p = float(perturb_p)
        self.mode = PERT_MODES[perturb_mode] if self.p > 0 else PERT_NONE
        self.r_success, self.r_step, self.r_action, self.r_wrong = r_success, r_step, r_action, r_wrong
        self.rng = random.Random(seed)
        self.state = 0
        self.target_attractor_id = 0
        self.state_attractor_id = 0
        self.n_steps = 0
        a = len(self.all_attractors)
        self.pair_weights = [[0.0 if (i == j and a > 1) else 1.0 for j in range(a)] for i in range(a)]

    # -- gym API ------------------------------------------------------------------
    def reset(self, seed: Optional[int] = None):
        if seed is not None:
            self.rng = random.Random(seed)
        a = len(self.all_attractors)
        pairs = [(i, j) for i in range(a) for j in range(a)]
        weights = [self.pair_weights[i][j] for i, j in pairs]
        src, tgt = self.rng.choices(pairs, weights=weights)[0]
        attr = self.all_attractors[src]
        self.state = bits_to_int(attr[self.rng.randrange(len(attr))])
        self.state_attractor_id, self.target_attractor_id = src, tgt
        self.n_steps = 0
        return (self.render(), self.target_state()), {}

    def target_state(self):
        return tuple(0 if b == "*" else int(b) for b in self.all_attractors[self.target_attractor_id][0])

    def render(self):
        return int_to_bits(self.state, self.n)

    def step(self, action):
        if isinstance(action, (int, np.integer)):
            action = [int(action)]
        actions = [int(a) for a in action]
        flip = flip_mask_from_actions(actions, self.n)
        sel = []
        for i in range(self.n):
            ps = self.net.probs[i]
            if len(ps) == 1:
                sel.append(0)
                continue
            u, acc, k = self.rng.random(), 0.0, 0
            for k, pk in enumerate(ps):
                acc += pk
                if u < acc:
                    break
            sel.append(k)
        pert = 0
        if self.mode != PERT_NONE:
            for i in range(self.n):
                if self.rng.random() < self.p:
                    pert |= 1 << i
        self.state = self.net.transition(self.state, flip, sel, pert, self.mode)
        self.n_steps += 1
        state = self.render()
        hit = self.in_target(state)
        truncated = (not hit) and self.horizon > 0 and self.n_steps >= self.horizon
        wrong = (not hit) and self.r_wrong != 0 and any(
            a != self.target_attractor_id and attractor_contains(at, state) for a, at in enumerate(self.all_attractors))
        reward = float(reward_f32(bin(flip).count("1"), hit, self.r_success, self.r_step, self.r_action, wrong, self.r_wrong))
        return state, reward, bool(hit), bool(truncated), {}

    # -- extras the reference calls (SURVEY.md 8a-6..8) ------------------------------
    def setTarget(self, attractor):
        attractor = list(map(tuple, attractor))
        self.target_attractor_id = self.all_attractors.index(attractor)

    def in_target(self, state) -> bool:
        return attractor_contains(self.all_attractors[self.target_attractor_id], state)

    def is_attracting_state(self, state) -> bool:
        return any(attractor_contains(a, state) for a in self.all_attractors)

    def set_state(self, state):
        self.state = bits_to_int(state)


# --------------------------------------------------------------------------------------
# Batched restatement of one env step with the kernels' own Philox streams
# (include/pbn_b200.h "Random streams"): bit-exact CPU twin of pbn_step().
# --------------------------------------------------------------------------------------

def survival_table(p: float, n: int) -> np.ndarray:
    """S[j] = floor((1-p)^j * 2^32) for j = 0..n, clamped to 2^32-1 (u32).  S[0] saturates."""
    out = np.zeros(n + 1, dtype=np.uint32)
    for j in range(n + 1):
        out[j] = min(int(((1.0 - p) ** j) * 4294967296.0), 0xFFFFFFFF)
    return out


def selection_thresholds(probs: Sequence[float]) -> List[int]:
    acc, out = 0.0, []
    for k, p in enumerate(probs):
        acc += p
        out.append(0xFFFFFFFF if k == len(probs) - 1 else min(int(round(acc * 4294967296.0)), 0xFFFFFFFF))
    return out


def _ctr(env_ids: np.ndarray, step_ctr: int, kind: int, idx: int):
    c0 = env_ids & np.uint64(0xFFFFFFFF)
    c1 = env_ids >> np.uint64(32)
    c2 = np.uint64(step_ctr & 0xFFFFFFFF)
    c3 = np.uint64(((step_ctr >> 32) & 0xFFFF) | (((kind << 12) | idx) << 16))
    return c0, c1, c2, c3


def scalar_stream_selection(net: OracleNetwork, env_ids: np.ndarray, step_ctr: int, seed: int) -> np.ndarray:
    """sel[E,N] as drawn by the thread-per-env kernel: gene i uses word i&3 of block (KIND_SELECT, i>>2);
    sel = number of cumulative thresholds <= u (last threshold excluded)."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    e = env_ids.shape[0]
    sel = np.zeros((e, net.n), dtype=np.uint8)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    for blk in range((net.n + 3) // 4):
        words = philox4x32(*_ctr(env_ids, step_ctr, KIND_SELECT, blk), k0, k1)
        for j in range(4):
            i = blk * 4 + j
            if i >= net.n:
                break
            thr = selection_thresholds(net.probs[i])[:-1]
            u = words[j].astype(np.uint64)
            s = np.zeros(e, dtype=np.uint8)
            for th in thr:
                s += (u >= np.uint64(th)).astype(np.uint8)
            sel[:, i] = s
    return sel


def scalar_stream_perturbation(n: int, p: float, env_ids: np.ndarray, step_ctr: int, seed: int) -> np.ndarray:
    """pert[E,W] by geometric skipping over the survival table (one u32 per perturbed gene + 1)."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    e = env_ids.shape[0]
    w = 1 if n <= 64 else 2
    pert = np.zeros((e, w), dtype=np.uint64)
    if p <= 0:
        return pert
    surv = survival_table(p, n).astype(np.uint64)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    pos = np.full(e, -1, dtype=np.int64)
    active = np.ones(e, dtype=bool)
    draw = 0
    while active.any():
        words = philox4x32(*_ctr(env_ids, step_ctr, KIND_PERTURB, draw >> 2), k0, k1)
        u = words[draw & 3].astype(np.uint64)
        skip = np.zeros(e, dtype=np.int64)
        for j in range(1, n + 1):
            skip += (u < surv[j]).astype(np.int64)
        pos = np.where(active, pos + skip + 1, pos)
        hit = active & (pos < n)
        idx = np.where(hit)[0]
        for wd in range(w):
            m = hit & ((pos >> 6) == wd)
            pert[m, wd] |= np.uint64(1) << (pos[m] & 63).astype(np.uint64)
        del idx
        active = hit
        draw += 1
    return pert


def batched_step(net: OracleNetwork, tables, words, actions, target_id, t, *, horizon, mode, sel, pert,
                 r_success, r_step, r_action, r_wrong=0.0):
    """One env step for E instances given sel[E,N] and pert[E,W] (injected or stream-drawn).
    Returns (next_words, t_next, reward, terminated, truncated).  Mirrors include/pbn_b200.h."""
    offs, care, val = tables
    words = np.asarray(words, dtype=np.uint64).reshape(-1, net.words)
    e = words.shape[0]
    actions = np.asarray(actions).reshape(e, -1).astype(np.int64)
    flip = np.zeros_like(words)
    for j in range(actions.shape[1]):
        a = actions[:, j]
        ok = (a >= 1) & (a <= net.n)
        g = np.where(ok, a - 1, 0)
        for wd in range(net.words):
            m = ok & ((g >> 6) == wd)
            flip[m, wd] |= np.uint64(1) << (g[m] & 63).astype(np.uint64)
    nflips = np.zeros(e, dtype=np.int64)
    for wd in range(net.words):
        nflips += np.array([bin(int(x)).count("1") for x in flip[:, wd]], dtype=np.int64) if e < 65536 else \
            _popcount64(flip[:, wd])
    nxt = net.transition_batch(words, flip, sel, pert, mode)
    target_id = np.asarray(target_id, dtype=np.int64)
    hit = np.zeros(e, dtype=bool)
    n_attr = len(offs) - 1
    for a in range(n_attr):
        m = target_id == a
        if not m.any():
            continue
        h = np.zeros(int(m.sum()), dtype=bool)
        for s in range(offs[a], offs[a + 1]):
            h |= ((nxt[m] & care[s]) == val[s]).all(axis=1)
        hit[m] = h
    t_next = np.minimum(np.asarray(t, dtype=np.int64) + 1, 65535).astype(np.uint16)
    trunc = (~hit) & (horizon > 0) & (t_next >= horizon)
    base = np.float32(r_step) + np.float32(r_action) * nflips.astype(np.float32)
    bonus = np.where(hit, np.float32(r_success), np.float32(0.0)).astype(np.float32)
    if r_wrong != 0.0:
        # the step ended in an attractor that is not the target ("wrong attractor")
        other = np.zeros(e, dtype=bool)
        for a in range(n_attr):
            m = (~hit) & (target_id != a)
            if not m.any():
                continue
            h = np.zeros(int(m.sum()), dtype=bool)
            for s in range(offs[a], offs[a + 1]):
                h |= ((nxt[m] & care[s]) == val[s]).all(axis=1)
            other[m] |= h
        bonus = np.where(other, np.float32(r_wrong), bonus).astype(np.float32)
    reward = (base + bonus).astype(np.float32)
    return nxt, t_next, reward, hit.astype(np.uint8), trunc.astype(np.uint8)


def _popcount64(x: np.ndarray) -> np.ndarray:
    x = x.astype(np.uint64)
    c = np.zeros(x.shape, dtype=np.int64)
    for sh in range(0, 64, 8):
        c += _POP8[((x >> np.uint64(sh)) & np.uint64(0xFF)).astype(np.int64)]
    return c


_POP8 = np.array([bin(i).count("1") for i in range(256)], dtype=np.int64)


def stream_reset(tables, n_attr: int, env_ids: np.ndarray, step_ctr: int, seed: int, pair_cum=None):
    """CPU twin of pbn_reset / the auto-reset of pbn_step: returns (state_words[E,W], source, target).
    Block (KIND_RESET, 0): word 0 picks the (source, target) pair, word 1 the state inside the
    source attractor (mul-hi), wildcards read as 0."""
    offs, care, val = tables
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    r = philox4x32(*_ctr(env_ids, step_ctr, KIND_RESET, 0), k0, k1)
    u0, u1 = r[0].astype(np.uint64), r[1].astype(np.uint64)
    a = n_attr
    if pair_cum is not None:
        pc = np.asarray(pair_cum, dtype=np.uint64)
        nz = [k for k in range(a * a) if pc[k] > (pc[k - 1] if k else 0) or (k == 0 and pc[0] > 0)]
        last = nz[-1] if nz else 0
        pair = (pc[None, : a * a - 1] <= u0[:, None]).sum(axis=1)
        pair = np.minimum(pair, last)
        src = pair // a
        tgt = pair - src * a
    elif a > 1:
        q = (u0 * np.uint64(a * (a - 1))) >> np.uint64(32)
        src = (q // np.uint64(a - 1)).astype(np.int64)
        tt = (q - src.astype(np.uint64) * np.uint64(a - 1)).astype(np.int64)
        tgt = tt + (tt >= src)
    else:
        src = np.zeros(len(env_ids), dtype=np.int64)
        tgt = np.zeros(len(env_ids), dtype=np.int64)
    src = np.asarray(src, dtype=np.int64)
    tgt = np.asarray(tgt, dtype=np.int64)
    o0 = offs[src].astype(np.int64)
    ns = (offs[src + 1] - offs[src]).astype(np.uint64)
    j = o0 + ((u1 * ns) >> np.uint64(32)).astype(np.int64)
    return val[j], src.astype(np.int32), tgt.astype(np.int32)


# --------------------------------------------------------------------------------------
# Sliced kernel streams (pbn_rl_b200/csrc/step_sliced.cuh, DESIGN.md "Sliced random stream")
# --------------------------------------------------------------------------------------

KIND_FIX = 3


def sliced_coords(env_ids: np.ndarray):
    """global env id -> (slice-group id, slice bit)."""
    e = np.asarray(env_ids, dtype=np.uint64)
    gid = ((e >> np.uint64(10)) << np.uint64(5)) | ((e >> np.uint64(2)) & np.uint64(31))
    bit = (((e >> np.uint64(7)) & np.uint64(7)) << np.uint64(2)) | (e & np.uint64(3))
    return gid, bit.astype(np.int64)


def sliced_survival(p: float, n: int) -> np.ndarray:
    """Survival table of one (column, warp) perturbation sub-stream: 8 rows x n genes."""
    slots = 8 * n
    out = np.zeros(slots + 1, dtype=np.uint64)
    for j in range(slots + 1):
        out[j] = min(int(((1.0 - p) ** j) * 4294967296.0), 0xFFFFFFFF)
    return out


def perturb_block(q: int, i: int) -> int:
    """Block index of block i of perturbation sub-stream q: 64q + i for the first 64 blocks, then 256 + 192q + (i - 64)
    (a walk over 8N slots draws up to 8N + 1 words, so the stream never reuses a word)."""
    return 64 * q + i if i < 64 else 256 + 192 * q + (i - 64)


class _WordStream:
    """Sequential 32-bit words of one (group, step, kind, sub-stream q) stream: blocks perturb_block(q, i)."""

    def __init__(self, gid, step_ctr, kind, k0, k1, q=0, first_word=0):
        self.gid, self.step, self.kind, self.k0, self.k1, self.q = gid, step_ctr, kind, k0, k1, q
        self.next = first_word
        self.blk = None

    def word(self):
        if (self.next & 3) == 0 or self.blk is None:
            r = philox4x32(*_ctr(np.array([self.gid], dtype=np.uint64), self.step, self.kind,
                                 perturb_block(self.q, self.next >> 2)), self.k0, self.k1)
            self.blk = [int(x[0]) for x in r]
        w = self.blk[self.next & 3]
        self.next += 1
        return w


def sliced_stream(net: OracleNetwork, p: float, env_ids: np.ndarray, step_ctr: int, seed: int):
    """(sel[E,N], pert[E,W]) exactly as the sliced kernel draws them for the given global env ids."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    e = env_ids.shape[0]
    n = net.n
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    gid, bit = sliced_coords(env_ids)
    groups, inv = np.unique(gid, return_inverse=True)
    ng = len(groups)
    ks = [len(ps) for ps in net.probs]
    full = np.uint64(0xFFFFFFFF)
    s0 = np.zeros((ng, n), dtype=np.uint64)
    s1 = np.zeros((ng, n), dtype=np.uint64)
    s2 = np.zeros((ng, n), dtype=np.uint64)   # third selection plane: genes with 5..8 predictors
    slot_gene = [i for i, k in enumerate(ks) if k > 1]
    # SELECT: slot r (the r-th gene with K > 1) owns block (SELECT, r) = words x, y, z, w.  K=2: s0 = x; K=4: (s0, s1) =
    # (x, y); K=3: the pairs (x, y), (z, w) -- pair value 3 is rejected and replaced by the next pair.
    weighted = {}
    for i, k in enumerate(ks):
        thr = selection_thresholds(net.probs[i])[:-1]
        # more than 4 predictors: always by threshold comparison (the pair-plane draw covers 2, 3 and 4)
        weighted[i] = k > 4 or any(abs(t - int(np.floor((j + 1) / k * 4294967296.0 + 0.5))) > 2 for j, t in enumerate(thr))
    for r, i in enumerate(slot_gene):
        if weighted[i]:
            # arbitrary probabilities: a 32-bit uniform per env, bit 31 - j of the column's envs = word j of the blocks
            # (SELECT, 128 + 8 r + i'), compared with the 32-bit thresholds: sel = #{k : cum[k] <= u}
            u32 = [np.zeros(ng, dtype=np.uint64) for _ in range(32)]   # per bit position b: the env's u
            for blk in range(8):
                words = philox4x32(*_ctr(groups, step_ctr, KIND_SELECT, 128 + 8 * r + blk), k0, k1)
                for j in range(4):
                    plane = words[j].astype(np.uint64)
                    for b in range(32):
                        u32[b] |= ((plane >> np.uint64(b)) & np.uint64(1)) << np.uint64(31 - (4 * blk + j))
            thr = selection_thresholds(net.probs[i])[:-1]
            for b in range(32):
                sel_b = np.zeros(ng, dtype=np.uint64)
                for t in thr:
                    sel_b += (u32[b] >= np.uint64(t)).astype(np.uint64)
                s0[:, i] |= (sel_b & np.uint64(1)) << np.uint64(b)
                s1[:, i] |= ((sel_b >> np.uint64(1)) & np.uint64(1)) << np.uint64(b)
                s2[:, i] |= ((sel_b >> np.uint64(2)) & np.uint64(1)) << np.uint64(b)
            continue
        x, y, z, w = (v.astype(np.uint64) for v in philox4x32(*_ctr(groups, step_ctr, KIND_SELECT, r), k0, k1))
        if ks[i] == 2:
            s0[:, i] = x
        elif ks[i] == 4:
            s0[:, i], s1[:, i] = x, y
        elif ks[i] == 3:
            rj = x & y
            s0[:, i] = (x & ~rj & full) | (z & rj)
            s1[:, i] = (y & ~rj & full) | (w & rj)
        else:
            raise ValueError("the sliced kernel takes 1..8 predictors per gene")
    # Pool of group q = r mod 4: blocks (FIX, 1024 q + i), i = 0, 1, ...; each block is two pair-planes (x, y), (z, w).
    # Per pair-plane the group's K=3 slots, in slot order, take bit b if they are still at value 3 there and no
    # earlier slot of the group has claimed bit b of this plane.  Blocks are consumed until no slot of the group is
    # at 3 anywhere in the column (columns that are done ignore further blocks).
    for q in range(4):
        slots_q = [i for r, i in enumerate(slot_gene) if r % 4 == q and ks[i] == 3 and not weighted[i]]
        if not slots_q:
            continue
        for it in range(1024):
            rej_any = np.zeros(ng, dtype=np.uint64)
            for i in slots_q:
                rej_any |= s0[:, i] & s1[:, i]
            act = np.nonzero(rej_any)[0]
            if len(act) == 0:
                break
            blk = [v.astype(np.uint64) for v in philox4x32(*_ctr(groups[act], step_ctr, KIND_FIX, 1024 * q + it), k0, k1)]
            for px, py in ((blk[0], blk[1]), (blk[2], blk[3])):
                av = np.full(len(act), full, dtype=np.uint64)
                for i in slots_q:
                    rj = s0[act, i] & s1[act, i]
                    tk = rj & av
                    av &= ~rj & full
                    s0[act, i] = (s0[act, i] & ~tk & full) | (px & tk)
                    s1[act, i] = (s1[act, i] & ~tk & full) | (py & tk)
    sh = bit.astype(np.uint64)[:, None]
    sel = (((s0[inv] >> sh) & np.uint64(1)) + 2 * ((s1[inv] >> sh) & np.uint64(1)) + 4 * ((s2[inv] >> sh) & np.uint64(1))).astype(np.uint8)
    for i, k in enumerate(ks):
        if k == 1:
            sel[:, i] = 0
    # perturbation events per group
    wds = 1 if n <= 64 else 2
    pert = np.zeros((e, wds), dtype=np.uint64)
    if p > 0:
        surv = sliced_survival(p, n)
        slots = 8 * n
        planes = np.zeros((ng, n), dtype=np.uint64)
        for g in range(ng):
            for q in range(4):  # sub-stream q covers slice bits 8q..8q+7
                ws = _WordStream(int(groups[g]), step_ctr, KIND_PERTURB, k0, k1, q)
                pos = -1
                while True:
                    u = ws.word()
                    skip = int(np.searchsorted(-surv[1:].astype(np.int64), -u, side="left"))  # #{j>=1: u < S[j]}
                    pos += skip + 1
                    if pos >= slots:
                        break
                    planes[g, pos >> 3] |= np.uint64(1) << np.uint64(8 * q + (pos & 7))
        pb = ((planes[inv] >> sh) & np.uint64(1))
        for i in range(n):
            pert[:, i >> 6] |= pb[:, i] << np.uint64(i & 63)
    return sel, pert
