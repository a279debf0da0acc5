"""Exact optimal control of small networks: finite-horizon dynamic programming over every state on the device.

The env is a finite Markov decision process, so for networks of at most ``PBN_DP_MAX_GENES`` = 28 genes the best
possible policy of a target attractor can be computed exactly by backward induction over all ``2^N`` states.  This is
the classical way to control a PBN and the yardstick an agent's scores are compared against: the optimal expected
return for every state and every number of steps left, the optimal flip set for each, and the exact value of any other
policy (a trained agent tabulated over all states).

One backup is two device operators of the C ABI (include/pbn_b200.h, "Exact optimal control") plus elementwise torch:

    Q_k(s, m) = r_step + r_action |m| + (P U_k)(s ^ m)        pbn_dp_expect:  W = P U
    V_k(s)    = max_m Q_k(s, m)                               pbn_dp_improve: max over the allowed flip sets
    U_k(t)    = r_success hit(t) + r_wrong wrong(t) + gamma (1 - hit(t)) V_{k-1}(t)

``hit`` / ``wrong`` are the step's classification of the next state against the target (pbn_in_target /
pbn_attractor_id over all states).  Objectives:

- ``"return"``: the env's own rewards, ``stages = env.horizon``, ``V_0 = 0``; ``V_H(s)`` is the optimal expected
  episode return from ``s`` at ``t = 0``.
- ``"steps"``: the ``model_tester`` / :func:`~pbn_rl_b200.evaluate.evaluate_all_pairs` step count: ``r_step = -1``,
  no other reward, ``gamma = 1``, ``stages = max_steps``, ``V_0 = -1`` off the target (a failure books
  ``max_steps + 1``) and target states worth 0, so ``-V(rep_source)`` is the expected ``matrix[source, target] / runs``.

Flip masks are ints with bit ``i`` = gene ``i`` (held in int32 tensors; ``N <= 28`` keeps them non-negative).
``policies[k - 1]`` and ``values[k]`` belong to ``k`` steps left.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, Dict, Mapping, Optional, Sequence, Union

import numpy as np
import torch

from . import _cabi
from ._cabi import check
from .vec_env import VecPBNEnv

__all__ = ["ControlSolution", "solve_control", "TabularPolicy", "policy_values", "tabulate_policy",
           "expected_all_pairs", "OBJECTIVES"]

OBJECTIVES = ("return", "steps")
_CHUNK = 1 << 22


def _vec(env) -> VecPBNEnv:
    """The :class:`VecPBNEnv` behind ``env`` (a ``PBNEnv`` / ``ControlPBNEnv`` through its ``.vec``)."""
    vec = getattr(env, "vec", env)
    if not isinstance(vec, VecPBNEnv):
        raise TypeError("expected a VecPBNEnv or a PBNEnv, got %r" % type(env).__name__)
    return vec


def _f32(x: float) -> float:
    """The fp32 value the env's reward arithmetic uses."""
    return float(np.float32(x))


def _popcount(m: torch.Tensor, n: int) -> torch.Tensor:
    sh = torch.arange(n, device=m.device, dtype=torch.int32)
    return ((m.to(torch.int32).unsqueeze(-1) >> sh) & 1).sum(-1)


def _state_index(words) -> torch.Tensor:
    t = torch.as_tensor(words)
    if t.dim() == 2:
        t = t[:, 0]
    return t.to(torch.int64)


def _bits_to_index(bits: torch.Tensor) -> torch.Tensor:
    """``[E, N]`` 0/1 (any dtype) -> ``[E]`` int64 state index."""
    n = bits.shape[-1]
    w = torch.ones(n, dtype=torch.int64, device=bits.device) << torch.arange(n, device=bits.device, dtype=torch.int64)
    return ((bits != 0).to(torch.int64) * w).sum(-1)


def _mask_to_actions(mask: torch.Tensor, n: int, bins: int) -> torch.Tensor:
    """Flip masks ``[E]`` -> uint8 actions ``[E, bins]``: the mask's genes + 1 in ascending order, 0-padded."""
    sh = torch.arange(n, device=mask.device, dtype=torch.int32)
    bit = ((mask.to(torch.int32).unsqueeze(-1) >> sh) & 1).bool()
    rank = torch.cumsum(bit.to(torch.int32), dim=1)
    gene = (sh + 1).unsqueeze(0)
    cols = [torch.where(bit & (rank == k + 1), gene, torch.zeros_like(gene)).sum(dim=1) for k in range(bins)]
    return torch.stack(cols, dim=1).to(torch.uint8)


def _actions_to_mask(actions: torch.Tensor, n: int) -> torch.Tensor:
    """uint8 actions ``[E, bins]`` -> flip masks ``[E]`` int32 (0 and values > N are no-ops, duplicates do not cancel)."""
    a = actions.to(torch.int64)
    ok = (a >= 1) & (a <= n)
    bits = torch.where(ok, torch.ones_like(a) << (a - 1).clamp(min=0), torch.zeros_like(a))
    m = torch.zeros(a.shape[0], dtype=torch.int64, device=a.device)
    for j in range(a.shape[1]):
        m |= bits[:, j]
    return m.to(torch.int32)


class _Backup:
    """Device buffers and the two operators of one env's backups."""

    def __init__(self, vec: VecPBNEnv):
        self.vec = vec
        self.n = vec.n_genes
        if self.n > _cabi.DP_MAX_GENES:
            raise _cabi.PbnError(_cabi.PBN_ERR_UNSUPPORTED, "exact control covers at most %d genes, the network has %d"
                                 % (_cabi.DP_MAX_GENES, self.n))
        self.S = 1 << self.n
        self.dev = vec.device
        self.lib, self.h = vec.lib, vec._h
        nbytes = int(self.lib.pbn_dp_workspace_bytes(self.h))
        if nbytes < 0:
            check(nbytes)
        self.ws = torch.empty((nbytes,), dtype=torch.uint8, device=self.dev)
        prob = [p for ps in vec.network.probabilities for p in ps]
        self.func_prob = torch.tensor(prob, dtype=torch.float64, device=self.dev)

    def expect(self, u: torch.Tensor) -> torch.Tensor:
        u = u.to(torch.float64).contiguous()
        w = torch.empty_like(u)
        check(self.lib.pbn_dp_expect(self.h, self.func_prob.data_ptr(), u.data_ptr(), w.data_ptr(), self.ws.data_ptr(),
                                     self.vec._stream()))
        return w

    def push(self, x: torch.Tensor, masks: Optional[torch.Tensor] = None) -> torch.Tensor:
        """y = x P, the forward operator of :meth:`expect` (x P_mu with flip masks ``masks`` [2^N] applied first).
        ``x`` must be a probability or sub-probability vector (pbn_dp_push's fixed point)."""
        x = x.to(torch.float64).contiguous()
        y = torch.empty_like(x)
        m = None if masks is None else masks.to(torch.int32).contiguous()
        check(self.lib.pbn_dp_push(self.h, self.func_prob.data_ptr(), x.data_ptr(), None if m is None else m.data_ptr(),
                                   y.data_ptr(), self.ws.data_ptr(), self.vec._stream()))
        return y

    def improve(self, w: torch.Tensor, flip_genes: int, max_flips: int, r_action: float):
        v = torch.empty_like(w)
        pol = torch.empty((self.S,), dtype=torch.int32, device=self.dev)
        check(self.lib.pbn_dp_improve(self.h, w.data_ptr(), int(flip_genes), int(max_flips), float(r_action),
                                      v.data_ptr(), pol.data_ptr(), self.ws.data_ptr(), self.vec._stream()))
        return v, pol

    def classify(self, target: int):
        """(hit, wrong) over all states: in the target attractor; in another attractor and not in the target."""
        vec = self.vec
        if vec.attractors is None:
            raise ValueError("the env has no attractor table")
        if not 0 <= int(target) < len(vec.attractors):
            raise ValueError("target %d outside 0..%d" % (target, len(vec.attractors) - 1))
        hit = torch.empty((self.S,), dtype=torch.uint8, device=self.dev)
        aid = torch.empty((self.S,), dtype=torch.int32, device=self.dev)
        for s0 in range(0, self.S, _CHUNK):
            n = min(_CHUNK, self.S - s0)
            st = torch.arange(s0, s0 + n, dtype=torch.int64, device=self.dev)
            tg = torch.full((n,), int(target), dtype=torch.int32, device=self.dev)
            check(self.lib.pbn_in_target(self.h, st.data_ptr(), tg.data_ptr(), hit[s0:].data_ptr(), n, vec._stream()))
            check(self.lib.pbn_attractor_id(self.h, st.data_ptr(), aid[s0:].data_ptr(), n, vec._stream()))
        hit = hit.bool()
        return hit, (~hit) & (aid >= 0)


@dataclass
class _Objective:
    stages: int
    gamma: float
    r_success: float
    r_step: float
    r_action: float
    r_wrong: float
    steps: bool


def _objective(vec: VecPBNEnv, objective: str, stages: Optional[int], gamma: float) -> _Objective:
    if objective == "return":
        st = vec.horizon if stages is None else int(stages)
        if st < 1:
            raise ValueError("the 'return' objective needs stages >= 1 (the env's horizon is %d)" % vec.horizon)
        return _Objective(st, float(gamma), _f32(vec.r_success), _f32(vec.r_step), _f32(vec.r_action),
                          _f32(vec.r_wrong), False)
    if objective == "steps":
        st = 100 if stages is None else int(stages)
        if st < 1:
            raise ValueError("stages must be >= 1")
        return _Objective(st, 1.0, 0.0, -1.0, 0.0, 0.0, True)
    raise ValueError("objective %r not in %r" % (objective, OBJECTIVES))


def _initial(obj: _Objective, hit: torch.Tensor) -> torch.Tensor:
    if obj.steps:
        return torch.where(hit, 0.0, -1.0).to(torch.float64)
    return torch.zeros(hit.shape, dtype=torch.float64, device=hit.device)


def _continuation(obj: _Objective, hit: torch.Tensor, wrong: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """U(t) = r_success hit + r_wrong wrong + gamma (1 - hit) V(t)."""
    base = torch.where(hit, obj.r_success, torch.where(wrong, obj.r_wrong, 0.0)).to(torch.float64)
    return base + torch.where(hit, 0.0, obj.gamma * v)


def _flip_set(env, vec: VecPBNEnv, flip_genes, max_flips):
    n = vec.n_genes
    control = getattr(env, "control_nodes", None)
    if flip_genes is None:
        genes = [c for c in control if 0 <= c < n] if control is not None else list(range(n))
        if max_flips is None:
            max_flips = len(genes) if control is not None else min(vec.bins, n)
    else:
        genes = [int(g) for g in flip_genes]
        if any(not 0 <= g < n for g in genes):
            raise ValueError("flip_genes must lie in [0, %d)" % n)
        if max_flips is None:
            max_flips = min(vec.bins, len(set(genes)))
    mask = 0
    for g in genes:
        mask |= 1 << g
    max_flips = int(max_flips)
    if not 0 <= max_flips <= vec.bins:
        raise ValueError("max_flips=%d outside 0..bins=%d (an action holds at most bins flips)" % (max_flips, vec.bins))
    return mask, max_flips


@dataclass
class ControlSolution:
    """The optimal finite-horizon policy of one target.  ``values[k]`` = ``V_k`` (``k`` steps left; fp64 ``[2^N]``),
    ``policies[k - 1]`` = its flip masks (int32 ``[2^N]``).  With ``keep_policies=False`` only the last stage is kept:
    ``values`` is ``[1, 2^N]`` and ``policies`` ``[1, 2^N]``."""

    target: int
    objective: str
    stages: int
    gamma: float
    flip_genes: int
    max_flips: int
    n_genes: int
    bins: int
    target_index: int                 # the target's representative state (first state, '*' -> 0)
    values: torch.Tensor
    policies: torch.Tensor
    full: bool = True

    def _stage(self, steps_left: Optional[int]) -> int:
        k = self.stages if steps_left is None else int(steps_left)
        if not 1 <= k <= self.stages:
            raise ValueError("steps_left=%d outside 1..%d" % (k, self.stages))
        if not self.full and k != self.stages:
            raise ValueError("only the last stage was kept (keep_policies=False)")
        return k

    def value(self, state_words, steps_left: Optional[int] = None) -> torch.Tensor:
        """Optimal value of the given states (packed words ``[E, 1]`` or indices ``[E]``) with ``steps_left`` steps."""
        k = self._stage(steps_left)
        idx = _state_index(state_words).to(self.values.device)
        return self.values[k if self.full else 0][idx]

    def masks(self, state_words, steps_left: Optional[int] = None) -> torch.Tensor:
        k = self._stage(steps_left)
        idx = _state_index(state_words).to(self.policies.device)
        return self.policies[k - 1 if self.full else 0][idx]

    def actions(self, state_words, steps_left: Optional[int] = None) -> torch.Tensor:
        """uint8 ``[E, bins]`` env actions of the optimal flip sets: the genes + 1 in ascending order, 0-padded."""
        return _mask_to_actions(self.masks(state_words, steps_left), self.n_genes, self.bins)


def solve_control(env, target: int, objective: str = "return", stages: Optional[int] = None, gamma: float = 1.0,
                  flip_genes: Optional[Sequence[int]] = None, max_flips: Optional[int] = None,
                  keep_policies: bool = True) -> ControlSolution:
    """Backward induction over all ``2^N`` states for ``target`` on ``env``'s device, with its dynamics (network,
    perturbation model and ``p``) and, for ``"return"``, its reward constants.  ``flip_genes`` defaults to every gene
    (a ``ControlPBNEnv``: its control nodes inside ``[0, N)``, ``max_flips = len`` of them), ``max_flips`` to the env's
    ``bins``.  See the module docstring for the objectives."""
    vec = _vec(env)
    obj = _objective(vec, objective, stages, gamma)
    mask, kmax = _flip_set(env, vec, flip_genes, max_flips)
    bk = _Backup(vec)
    hit, wrong = bk.classify(target)
    v = _initial(obj, hit)
    values, policies = [v], []
    for _ in range(obj.stages):
        w = bk.expect(_continuation(obj, hit, wrong, v))
        best, pol = bk.improve(w, mask, kmax, obj.r_action)
        v = obj.r_step + best
        if obj.steps:
            v = torch.where(hit, 0.0, v)
        if keep_policies:
            values.append(v)
            policies.append(pol)
    if not keep_policies:
        values, policies = [v], [pol]
    rep = vec.attractors.representative_words()[int(target)]
    return ControlSolution(int(target), objective, obj.stages, obj.gamma, mask, kmax, vec.n_genes, vec.bins,
                           int(rep[0]), torch.stack(values), torch.stack(policies), bool(keep_policies))


def policy_values(env, target: int, masks: torch.Tensor, objective: str = "return", stages: Optional[int] = None,
                  gamma: float = 1.0) -> torch.Tensor:
    """Exact values ``[stages + 1, 2^N]`` of a given policy: the recursion of :func:`solve_control` with the maximum
    replaced by ``V(s) = r_step + r_action |m(s)| + W[s ^ m(s)]``.  ``masks``: a stationary ``[2^N]`` flip-mask table
    (e.g. from :func:`tabulate_policy`) or one per stage, ``[stages, 2^N]`` with ``masks[k - 1]`` for ``k`` steps
    left."""
    vec = _vec(env)
    obj = _objective(vec, objective, stages, gamma)
    bk = _Backup(vec)
    m = torch.as_tensor(masks).to(device=bk.dev, dtype=torch.int64)
    if m.dim() == 1:
        m = m.unsqueeze(0).expand(obj.stages, -1)
    if m.shape != (obj.stages, bk.S):
        raise ValueError("masks must be [2^N] or [stages, 2^N] = [%d, %d]" % (obj.stages, bk.S))
    if ((m >> vec.n_genes) != 0).any():
        raise ValueError("masks flip genes beyond the network")
    hit, wrong = bk.classify(target)
    s = torch.arange(bk.S, device=bk.dev, dtype=torch.int64)
    v = _initial(obj, hit)
    out = [v]
    for k in range(1, obj.stages + 1):
        w = bk.expect(_continuation(obj, hit, wrong, v))
        mk = m[k - 1]
        v = obj.r_step + (obj.r_action * _popcount(mk, vec.n_genes).to(torch.float64) + w[s ^ mk])
        if obj.steps:
            v = torch.where(hit, 0.0, v)
        out.append(v)
    return torch.stack(out)


def tabulate_policy(policy: Callable[[torch.Tensor], torch.Tensor], env, target: int, chunk: int = 1 << 16) -> torch.Tensor:
    """The flip masks ``[2^N]`` (int32) an agent's policy chooses in every state: ``policy`` gets the float32
    ``[2, chunk, N]`` observation (state bits, target representative bits -- :meth:`VecPBNEnv.observe`'s layout) and
    returns uint8 actions ``[chunk, bins]``.  With :func:`policy_values` this gives a trained agent's exact value and
    its gap to the optimum."""
    vec = _vec(env)
    n = vec.n_genes
    if n > _cabi.DP_MAX_GENES:
        raise ValueError("exact control covers at most %d genes" % _cabi.DP_MAX_GENES)
    S, dev = 1 << n, vec.device
    rep = int(vec.attractors.representative_words()[int(target)][0])
    sh = torch.arange(n, device=dev, dtype=torch.int64)
    tgt_bits = ((torch.tensor(rep, device=dev) >> sh) & 1).to(torch.float32)
    out = torch.empty((S,), dtype=torch.int32, device=dev)
    for s0 in range(0, S, chunk):
        c = min(chunk, S - s0)
        st = torch.arange(s0, s0 + c, device=dev, dtype=torch.int64)
        obs = torch.empty((2, c, n), dtype=torch.float32, device=dev)
        obs[0] = ((st.unsqueeze(1) >> sh) & 1).to(torch.float32)
        obs[1] = tgt_bits
        act = torch.as_tensor(policy(obs)).to(dev)
        out[s0:s0 + c] = _actions_to_mask(act.reshape(c, -1), n)
    return out


class TabularPolicy:
    """A tabulated (e.g. optimal) policy with the :func:`~pbn_rl_b200.evaluate.evaluate_all_pairs` signature:
    ``policy(obs [2, E, N]) -> uint8 [E, bins]``.  The state bits of ``obs[0]`` index the tables; the target
    representative bits of ``obs[1]`` pick the target's solution.  It counts its calls to know the steps left
    (``stages - calls``, at least 1), so a fresh instance (or :meth:`reset`) runs one evaluation."""

    def __init__(self, solutions: Union[Mapping[int, ControlSolution], Sequence[ControlSolution]]):
        sols = list(solutions.values()) if isinstance(solutions, Mapping) else list(solutions)
        if not sols:
            raise ValueError("no solutions")
        stages = {s.stages for s in sols}
        if len(stages) != 1 or any(not s.full for s in sols):
            raise ValueError("the solutions must share their number of stages and keep every stage's policy")
        self.stages = stages.pop()
        self.n, self.bins = sols[0].n_genes, sols[0].bins
        dev = sols[0].policies.device
        self.table = torch.stack([s.policies for s in sols])                       # [T, stages, 2^N]
        self.reps = torch.tensor([s.target_index for s in sols], dtype=torch.int64, device=dev)
        self.calls = 0

    def reset(self) -> None:
        self.calls = 0

    def __call__(self, obs: torch.Tensor) -> torch.Tensor:
        k = max(self.stages - self.calls, 1)
        self.calls += 1
        s = _bits_to_index(obs[0])
        t = _bits_to_index(obs[1])
        match = t.unsqueeze(1) == self.reps.unsqueeze(0)                            # [E, T]
        if not bool(match.any(dim=1).all()):
            raise ValueError("an observation's target is not among the solved targets")
        slot = match.to(torch.int8).argmax(dim=1)
        m = self.table[slot, k - 1, s]
        return _mask_to_actions(m, self.n, self.bins)


def expected_all_pairs(env, attractors, solutions: Union[Mapping[int, ControlSolution], Sequence[ControlSolution]]) -> np.ndarray:
    """The exact expected ``model_tester`` matrix per run, ``[A, A]``: entry ``[s, t]`` = the optimal policy's expected
    step count from source ``s``'s representative state to target ``t`` (``"steps"`` solutions, one per target; the
    diagonal is 0 because every representative lies in its own attractor)."""
    sols = dict(solutions) if isinstance(solutions, Mapping) else {s.target: s for s in solutions}
    reps = attractors.representative_words()
    a = len(sols)
    out = np.zeros((a, a), dtype=np.float64)
    for t in range(a):
        sol = sols[t]
        if sol.objective != "steps":
            raise ValueError("expected_all_pairs needs 'steps' solutions")
        v = sol.value(torch.from_numpy(reps[:a, :1].astype(np.int64)))
        out[:, t] = (-v).cpu().numpy()
    return out
