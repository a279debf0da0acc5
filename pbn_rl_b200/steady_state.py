"""Exact state distributions of small networks: the forward operator ``x -> x P`` over every state on the device.

For networks of at most ``PBN_DP_MAX_GENES`` = 28 genes the distribution of the env's state after ``k`` steps, and the
steady-state distribution (SSD) ``pi = pi P`` of a perturbed network, can be computed exactly over all ``2^N``
states (Shmulevich et al.'s classical PBN analysis).  They are the yardstick of the sampled statistics of
:func:`~pbn_rl_b200.discover.steady_state_statistics`: how far a sampled SSD is from the truth, and how much burn-in a
network needs.

Each step is one ``pbn_dp_push`` (include/pbn_b200.h, "Exact optimal control"): ``y = x P``, or ``x P_mu`` with a
closed-loop policy's flip masks ``mu`` applied before the step (``P_mu(s, .) = P(s ^ mu(s), .)``, the env's step with
flips, as in :func:`~pbn_rl_b200.control.policy_values`).  The push sums in fixed point, so it is deterministic and
needs a probability or sub-probability vector (``x >= 0``, ``sum x <= 1``).  States are indices with bit ``i`` = gene
``i``.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Union

import numpy as np
import torch

from .control import _Backup, _vec

__all__ = ["StateDistribution", "propagate", "stationary_distribution"]


@dataclass
class StateDistribution:
    """A distribution over all ``2^N`` states: ``probs`` is the fp64 ``[2^N]`` device tensor (entry ``s`` = state
    ``s``).  :func:`stationary_distribution` fills in ``iterations`` (pushes run), ``residual`` (the L1 change of the
    last checked iteration) and ``converged``; :func:`propagate` sets ``steps``.  The summaries reduce with reshapes and
    sums (no atomics), so they are deterministic."""

    probs: torch.Tensor
    n_genes: int
    steps: int = 0
    iterations: int = 0
    residual: float = float("nan")
    converged: bool = False

    def marginals(self) -> np.ndarray:
        """P(gene g is ON), float64 ``[N]`` (the layout of :meth:`StateRecorder.marginals`)."""
        n, x = self.n_genes, self.probs
        return np.array([float(x.view(1 << (n - 1 - g), 2, 1 << g)[:, 1, :].sum()) for g in range(n)])

    def projection(self, genes: Sequence[int]) -> np.ndarray:
        """The distribution of the states projected onto ``genes`` (any number of distinct genes), float64
        ``[2^len(genes)]`` with bin bit j = gene ``genes[j]`` (the layout of :meth:`StateRecorder.distribution`)."""
        n = self.n_genes
        genes = [int(g) for g in genes]
        if len(set(genes)) != len(genes) or any(not 0 <= g < n for g in genes):
            raise ValueError("projection genes must be distinct and in [0, %d)" % n)
        # axis a of the [2] * N view is gene N - 1 - a
        v = self.probs.view([2] * n)
        drop = [n - 1 - g for g in range(n) if g not in genes]
        r = v.sum(dim=drop) if drop else v
        kept = sorted(genes, reverse=True)                   # gene order of r's axes
        r = r.permute([kept.index(g) for g in reversed(genes)]) if genes else r
        return r.reshape(-1).cpu().numpy()

    def mass(self, states) -> float:
        """The total probability of the listed states (indices, or packed words ``[E, W]``; each counted once)."""
        idx = _indices(states, self.n_genes).to(self.probs.device)
        return float(self.probs[torch.unique(idx)].sum())


def _indices(states, n: int) -> torch.Tensor:
    t = torch.as_tensor(states)
    if t.dim() == 2:
        t = t[:, 0]
    t = t.reshape(-1).to(torch.int64)
    if bool(((t < 0) | (t >= (1 << n))).any()):
        raise ValueError("states outside [0, 2^%d)" % n)
    return t


def _start(initial, n: int, dev) -> torch.Tensor:
    """A distribution ``[2^N]`` (floating point), or one state (an index, or its packed word ``[1]`` / ``[1, 1]``) as a
    point mass; validated once: ``x >= 0`` and ``sum x <= 1 + 1e-12``."""
    S = 1 << n
    t = torch.as_tensor(initial)
    if t.is_floating_point():
        if t.shape != (S,):
            raise ValueError("an initial distribution must be [2^N] = [%d], got %s" % (S, tuple(t.shape)))
        x = t.to(device=dev, dtype=torch.float64).contiguous()
        if bool((x < 0).any()) or not bool(torch.isfinite(x).all()):
            raise ValueError("an initial distribution must be finite and non-negative")
        total = float(x.sum())
        if total > 1.0 + 1e-12:
            raise ValueError("an initial distribution must have mass <= 1, got %.17g" % total)
        return x
    if t.numel() != 1:     # N <= 28: one packed word per state
        raise ValueError("an initial state must be one index or the packed words of one state")
    s = int(t.reshape(-1)[0])
    if not 0 <= s < S:
        raise ValueError("initial state %d outside [0, 2^%d)" % (s, n))
    x = torch.zeros(S, dtype=torch.float64, device=dev)
    x[s] = 1.0
    return x


def _masks(masks, n: int, dev) -> Optional[torch.Tensor]:
    if masks is None:
        return None
    m = torch.as_tensor(masks).to(device=dev, dtype=torch.int64)
    if m.shape != (1 << n,):
        raise ValueError("masks must be [2^N] = [%d]" % (1 << n))
    if bool(((m < 0) | ((m >> n) != 0)).any()):
        raise ValueError("masks flip genes beyond the %d of the network" % n)
    return m.to(torch.int32)


def propagate(env, initial, steps: int, masks=None, keep: bool = False) -> Union[StateDistribution, List[StateDistribution]]:
    """The exact distribution of ``env``'s state after ``steps`` steps from ``initial`` (a distribution ``[2^N]``, a
    state index, or packed words), with ``env``'s network, perturbation model and ``p`` (any ``p``, 0 included) and,
    with ``masks`` ``[2^N]``, the flips ``masks[s]`` applied in state ``s`` before each step.  ``keep=True`` returns the
    distributions after 0, 1, ..., ``steps`` steps."""
    vec = _vec(env)
    bk = _Backup(vec)
    if int(steps) < 0:
        raise ValueError("steps must be >= 0")
    x = _start(initial, bk.n, bk.dev)
    m = _masks(masks, bk.n, bk.dev)
    out = [StateDistribution(x, bk.n)] if keep else []
    for k in range(1, int(steps) + 1):
        x = bk.push(x, m)
        if keep:
            out.append(StateDistribution(x, bk.n, steps=k))
    return out if keep else StateDistribution(x, bk.n, steps=int(steps))


def stationary_distribution(env, tol: float = 1e-10, max_iters: int = 100000, initial=None, masks=None,
                            check_every: int = 16) -> StateDistribution:
    """The steady-state distribution ``pi = pi P`` of ``env``'s perturbed network (``pi P_mu`` with ``masks``) by
    power iteration from ``initial`` (default: uniform).  Every ``check_every`` pushes the L1 change of the last one,
    ``|x P - x|_1``, is compared with ``tol`` and the iterate is renormalised to mass 1 (which absorbs the fixed-point
    rounding of the push).

    With ``p > 0`` models A and B make the chain irreducible and aperiodic, so ``pi`` is unique and the iteration
    converges.  The residual bounds the error only up to the spectral gap, ``|x - pi|_1 <~ residual / gap`` with a gap
    of about ``N p`` for small ``p``: tighten ``tol`` accordingly.  ``p = 0`` is refused (the chain need not be ergodic
    and may cycle): use :func:`propagate` for the transient distribution there."""
    vec = _vec(env)
    if not vec.perturb_p > 0.0:
        raise ValueError("stationary_distribution needs perturbation (p > 0): without it the chain need not be ergodic "
                         "and may cycle; use propagate() for the distribution after a given number of steps")
    if int(check_every) < 1 or int(max_iters) < 1:
        raise ValueError("check_every and max_iters must be >= 1")
    bk = _Backup(vec)
    S = bk.S
    x = (torch.full((S,), 1.0 / S, dtype=torch.float64, device=bk.dev) if initial is None
         else _start(initial, bk.n, bk.dev))
    m = _masks(masks, bk.n, bk.dev)
    residual, it = float("nan"), 0
    while it < int(max_iters):
        y = bk.push(x, m)
        it += 1
        if it % int(check_every) == 0 or it == int(max_iters):
            residual = float((y - x).abs().sum())
            y = y / y.sum()
            if residual < tol:
                return StateDistribution(y, bk.n, iterations=it, residual=residual, converged=True)
        x = y
    return StateDistribution(x, bk.n, iterations=it, residual=residual, converged=False)
