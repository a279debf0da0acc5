"""Closed-form laws of one PBN step, of the reset, and the decision rule that compares sampled counts with them.

Written from the step contract (include/pbn_b200.h, "Random streams" aside), not from the kernels, the truth-table
compiler or the oracle's Philox twins: the selection step evaluates the OracleNetwork's Python expressions, and states
are Python ints, so every N <= 128 works.  fp64 throughout.

- ``q_genes(onet, s)``: q_i(s), the summed selection probability of gene i's predictors that yield 1 in state s.
- One-step law from (s, flips), s1 = s ^ flips, F the selection step (independent genes, gene i is 1 with q_i(s1)):
  none and B are F followed by the mask (product forms); C sets gene i to m_i ? not s1_i : f_i (again a product);
  A is c F + K_p - c delta_{s1}, c = (1 - p)^N, K_p the mask channel applied to s1.
- Marginals, projections onto up to 16 genes (A: c prod_G F_i + prod_G K_i - c delta(t_G = s1_G)) and full rows.
- Network builders: selection probes, keep and negate networks.
- The reset law: (source, target) uniform over ordered pairs with source != target, or proportional to the pair weights;
  the state uniform over the source attractor's entries, wildcards read as 0.
- ``Judge``: the decision rule.  A Bernoulli count c of n trials at probability r fails when its exact two-sided
  binomial tail, 2 min(P(X <= c), P(X >= c)), is below ``ALPHA`` = 1.97e-9, the two-sided Gaussian tail at
  ``Z_MAX`` = 6 sigma.  The exact tail keeps every check's false-alarm probability at or below ALPHA whatever n r is:
  the Gaussian rule |z| > 6 does not (2.3e-7 at n = 2^14, r = 0.001, a slice-bit cell of a rare predictor).  The z-score
  is still reported as the margin.  Chi-square tests (bins of expected count below 5 pooled into one) must have
  p > ``P_MIN`` = 1e-7, and a count in a bin of probability 0 fails at once.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import numpy as np

from oracle import pbn_oracle as O

Z_MAX = 6.0
ALPHA = 1.973175290075389e-09     # 2 * Q(Z_MAX), the two-sided normal tail at 6 sigma
P_MIN = 1e-7


# ---------------------------------------------------------------------------------------------- selection step
def _env_of(onet, s: int) -> Dict[str, bool]:
    return {g: bool((s >> i) & 1) for i, g in enumerate(onet.genes)}


def q_genes(onet, s: int) -> np.ndarray:
    """q_i(s) for every gene: each predictor expression evaluated by Python on the bits of the int ``s``."""
    env = _env_of(onet, s)
    q = np.zeros(onet.n)
    for i in range(onet.n):
        for code, p in zip(onet.py_code[i], onet.probs[i]):
            if eval(code, {}, env):
                q[i] += p
    return np.minimum(q, 1.0)


def q_states(onet, states: Sequence[int]) -> np.ndarray:
    """q_i(s) for many states at once ([len(states), N]); the same expressions in their numpy form."""
    bits = np.array([[(int(s) >> i) & 1 for i in range(onet.n)] for s in states], dtype=bool).reshape(-1, onet.n)
    ns = {g: bits[:, i] for i, g in enumerate(onet.genes)}
    q = np.zeros(bits.shape)
    for i in range(onet.n):
        for code, p in zip(onet.np_code[i], onet.probs[i]):
            q[:, i] += p * np.broadcast_to(np.asarray(eval(code, {}, ns), dtype=bool), (bits.shape[0],))
    return np.minimum(q, 1.0)


def free_genes(q: np.ndarray) -> List[int]:
    return [i for i, v in enumerate(q) if 0.0 < v < 1.0]


def _bit(s: int, i: int) -> int:
    return (s >> i) & 1


def gene_laws(onet, s: int, flips: int, mode, p: float):
    """The per-gene pieces of the step law: (s1, F, K, c) with F_i = P(f_i = 1) = q_i(s1), K_i = P((s1 ^ m)_i = 1) and
    c = (1 - p)^N.  For none/B/C the step law is the product of Bernoulli(marginals); for A it is c F + K - c delta."""
    mode = O.PERT_MODES[mode]
    s1 = s ^ flips
    F = q_genes(onet, s1)
    s1b = np.array([_bit(s1, i) for i in range(onet.n)], dtype=np.float64)
    K = np.where(s1b == 1, 1.0 - p, p)
    c = (1.0 - p) ** onet.n
    return s1, F, K, c, mode


def marginals(onet, s: int, flips: int, mode, p: float) -> np.ndarray:
    """P(gene i = 1 after the step)."""
    s1, F, K, c, mode = gene_laws(onet, s, flips, mode, p)
    s1b = np.array([_bit(s1, i) for i in range(onet.n)], dtype=np.float64)
    if mode == O.PERT_NONE or p == 0.0:
        return F
    if mode == O.PERT_B:
        return F * (1.0 - p) + (1.0 - F) * p
    if mode == O.PERT_C:
        return p * (1.0 - s1b) + (1.0 - p) * F
    return c * F + K - c * s1b


def product_law(r: Sequence[float]) -> np.ndarray:
    """Independent Bernoulli(r_j): array [2^len(r)], bin bit j = variable j."""
    out = np.ones(1)
    for v in r:
        out = np.concatenate([out * (1.0 - v), out * v])
    return out


def projection(onet, s: int, flips: int, mode, p: float, genes: Sequence[int]) -> np.ndarray:
    """The step law projected onto ``genes`` (bin bit j = gene genes[j]), up to 16 genes."""
    genes = list(genes)
    assert len(genes) <= 16
    s1, F, K, c, m = gene_laws(onet, s, flips, mode, p)
    if m != O.PERT_A or p == 0.0:
        return product_law(marginals(onet, s, flips, mode, p)[genes])
    out = c * product_law(F[genes]) + product_law(K[genes])
    out[sum(_bit(s1, g) << j for j, g in enumerate(genes))] -= c
    return np.maximum(out, 0.0)


def row_genes(onet, s: int, flips: int, mode, p: float) -> List[int]:
    """The genes the step can change the value of (the rest are fixed): the support of the full row."""
    r = marginals(onet, s, flips, mode, p)
    return [i for i, v in enumerate(r) if 0.0 < v < 1.0]


def full_row(onet, s: int, flips: int, mode, p: float):
    """(genes, law over them, fixed part): the full row of the step as the law of its free genes and the value of
    every other gene (certain).  The law is None when more than 16 genes are free."""
    genes = row_genes(onet, s, flips, mode, p)
    r = marginals(onet, s, flips, mode, p)
    fixed = sum(1 << i for i, v in enumerate(r) if v >= 1.0)
    return genes, (projection(onet, s, flips, mode, p, genes) if len(genes) <= 16 else None), fixed


def dense_matrix(onet, mode, p: float) -> np.ndarray:
    """P[s, t] over all 2^N states (N <= 10) from the full rows."""
    n = onet.n
    S = 1 << n
    P = np.zeros((S, S))
    for s in range(S):
        law = projection(onet, s, 0, mode, p, list(range(n)))
        P[s] = law
    return P


# ---------------------------------------------------------------------------------------------- network builders
def probe_network(layout: Sequence[Optional[Sequence[float]]], n_code: int):
    """Genes x0..x{n-1}.  The first ``n_code`` genes are code genes c_j = x_j that keep their value; ``layout[i]``
    (i >= n_code) is None for another gene that keeps its value, or a probability vector: probe gene i then has the
    predictors x_{c_0}, x_{c_1}, ... with those selection probabilities.  From the state where only c_j is on, probe
    gene i is 1 after the step exactly when it selected predictor j.  Returns (genes, exprs)."""
    n = len(layout)
    genes = ["x%d" % i for i in range(n)]
    exprs = []
    for i in range(n):
        probs = layout[i] if i >= n_code else None
        if probs is None:
            exprs.append([("x%d" % i, 1.0)])
        else:
            assert len(probs) <= n_code
            exprs.append([("x%d" % j, float(w)) for j, w in enumerate(probs)])
    return genes, exprs


def probe_law(layout, n_code: int) -> np.ndarray:
    """P(probe gene i = 1 | code state j) as [n_code, N] (0 for code genes and keep genes: they stay 0 or 1 as set)."""
    n = len(layout)
    out = np.zeros((n_code, n))
    for i in range(n_code, n):
        if layout[i] is not None:
            w = np.asarray(layout[i], dtype=np.float64)
            out[:len(w), i] = w / w.sum()
    for j in range(n_code):
        out[j, j] = 1.0
    return out


def keep_network(n: int):
    genes = ["x%d" % i for i in range(n)]
    return genes, [[("x%d" % i, 1.0)] for i in range(n)]


def negate_network(n: int):
    genes = ["x%d" % i for i in range(n)]
    return genes, [[("~ x%d" % i, 1.0)] for i in range(n)]


def binomial_pmf(n: int, p: float) -> np.ndarray:
    k = np.arange(n + 1)
    return np.array([math.comb(n, int(j)) for j in k], dtype=np.float64) * p ** k * (1.0 - p) ** (n - k)


def negate_flip_law(n: int, p: float) -> np.ndarray:
    """Negate network, model A: law of popcount(t ^ s).  A perturbed step lands on s ^ m (|m| >= 1); an unperturbed one
    on not s (N genes differ).  So 0 is impossible."""
    out = binomial_pmf(n, p)
    out[n] += out[0]
    out[0] = 0.0
    return out


# ---------------------------------------------------------------------------------------------- reset law
def reset_pair_law(n_attr: int, pair_weights=None) -> np.ndarray:
    """P(source, target) as [A * A] (index source * A + target)."""
    a = n_attr
    if pair_weights is not None:
        w = np.asarray(pair_weights, dtype=np.float64).reshape(-1)
        return w / w.sum()
    if a == 1:
        return np.ones(1)
    out = np.full((a, a), 1.0 / (a * (a - 1)))
    np.fill_diagonal(out, 0.0)
    return out.reshape(-1)


def reset_entries(attractors) -> List[List[int]]:
    """The state each entry of each attractor resets to: its bits with wildcards read as 0."""
    return [[O.bits_to_int(e) for e in attr] for attr in attractors]


def reset_law(attractors, pair_weights=None) -> np.ndarray:
    """Joint law of (source, target, entry) as [A, A, max entries]: pair law times uniform over the source's entries."""
    a = len(attractors)
    m = max(len(x) for x in attractors)
    pair = reset_pair_law(a, pair_weights).reshape(a, a)
    out = np.zeros((a, a, m))
    for src, attr in enumerate(attractors):
        out[src, :, :len(attr)] = pair[src][:, None] / len(attr)
    return out


# ---------------------------------------------------------------------------------------------- decision rule
def chi2_stat(counts, probs):
    """(statistic, degrees of freedom, impossible) of counts against probs: bins with expected count below 5 are pooled
    into one; ``impossible`` counts the samples that fell where the probability is 0."""
    counts = np.asarray(counts, dtype=np.float64).reshape(-1)
    probs = np.asarray(probs, dtype=np.float64).reshape(-1)
    total = counts.sum()
    impossible = float(counts[probs <= 0.0].sum())
    exp = probs / probs.sum() * total
    big = exp >= 5.0
    obs = counts[big]
    ex = exp[big]
    rest_o, rest_e = counts[~big].sum(), exp[~big].sum()
    if rest_e > 0.0:
        obs = np.append(obs, rest_o)
        ex = np.append(ex, rest_e)
    if ex.size < 2:
        return 0.0, 0, impossible
    return float(((obs - ex) ** 2 / ex).sum()), ex.size - 1, impossible


def chi2_p(tables) -> float:
    """p-value of the summed chi-square of independent tables [(counts, probs), ...]; 0 on an impossible count."""
    from scipy.stats import chi2
    stat, dof = 0.0, 0
    for counts, probs in tables:
        s, d, imp = chi2_stat(counts, probs)
        if imp:
            return 0.0
        stat += s
        dof += d
    return 1.0 if dof == 0 else float(chi2.sf(stat, dof))


def binomial_p(counts, totals, probs) -> np.ndarray:
    """Exact two-sided binomial tail 2 min(P(X <= c), P(X >= c)) (capped at 1) of Bernoulli counts; where r is 0 or 1
    any deviation has tail 0."""
    from scipy.stats import binom
    c = np.asarray(counts, dtype=np.float64)
    n = np.broadcast_to(np.asarray(totals, dtype=np.float64), c.shape)
    r = np.broadcast_to(np.asarray(probs, dtype=np.float64), c.shape)
    return np.minimum(1.0, 2.0 * np.minimum(binom.cdf(c, n, r), binom.sf(c - 1.0, n, r)))


def z_scores(counts, totals, probs) -> np.ndarray:
    """(count - n r) / sqrt(n r (1 - r)) of Bernoulli counts; where r is 0 or 1 any deviation is infinite."""
    c = np.asarray(counts, dtype=np.float64)
    n = np.broadcast_to(np.asarray(totals, dtype=np.float64), c.shape)
    r = np.broadcast_to(np.asarray(probs, dtype=np.float64), c.shape)
    var = n * r * (1.0 - r)
    dev = c - n * r
    with np.errstate(divide="ignore", invalid="ignore"):
        z = np.where(var > 0.0, dev / np.sqrt(np.where(var > 0.0, var, 1.0)),
                     np.where(np.abs(dev) > 0.5, np.inf, 0.0))
    return z


class Judge:
    """Collects the outcomes of one test's comparisons: failures, and the margins (smallest p-value, largest |z|)."""

    def __init__(self, name: str = ""):
        self.name = name
        self.failures: List[str] = []
        self.min_p = 1.0
        self.max_z = 0.0
        self.min_p_binom = 1.0
        self.n_z = 0
        self.n_chi2 = 0

    def z(self, counts, totals, probs, tag: str) -> float:
        """Bernoulli counts: fail where the exact binomial tail is below ALPHA; the largest |z| is the margin."""
        z = np.abs(z_scores(counts, totals, probs))
        pb = binomial_p(counts, totals, probs)
        self.n_z += z.size
        m = float(z.max()) if z.size else 0.0
        self.max_z = max(self.max_z, m)
        if z.size:
            self.min_p_binom = min(self.min_p_binom, float(pb.min()))
        if z.size and float(pb.min()) < ALPHA:
            at = np.unravel_index(int(np.argmin(pb)), pb.shape)
            self.failures.append("%s: binomial tail %.3g (|z| = %.2f) at %s" % (tag, float(pb[at]), float(z[at]),
                                                                              tuple(int(x) for x in at)))
        return m

    def chi2(self, tables, tag: str) -> float:
        if isinstance(tables, tuple):
            tables = [tables]
        p = chi2_p(tables)
        self.n_chi2 += 1
        self.min_p = min(self.min_p, p)
        if p < P_MIN:
            self.failures.append("%s: chi-square p = %.3g" % (tag, p))
        return p

    def exact(self, ok: bool, tag: str) -> None:
        if not ok:
            self.failures.append(tag)

    def report(self) -> str:
        return ("LAW %s: %d binomial tests, max |z| %.2f, min tail %.3g; %d chi-square tests, min p %.3g; %d failures"
                % (self.name, self.n_z, self.max_z, self.min_p_binom, self.n_chi2, self.min_p, len(self.failures)))

    def check(self) -> None:
        print(self.report())
        assert not self.failures, "\n".join(self.failures[:20])
