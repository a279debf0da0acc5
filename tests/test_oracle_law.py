"""CPU: the closed-form laws of tests/law_oracle.py against enumeration, and the power of its decision rule.

- One-step rows (none / A / B / C, with and without flips) against every (selection, perturbation mask) pair pushed
  through the oracle's deterministic step, weighted by its probability.
- Dense rows against control_oracle.transition_matrix (none / A / B).
- Projections against the marginalised full row; q_i(s) against control_oracle and at 128 genes.
- Calibration at the GPU sample size E = 2^22, fixed seeds: samples of the exact law pass; a predictor probability
  moved by 2^-7, p scaled by 1.05 and a two-step law that reuses step 1's selections are rejected.
- The exact false-alarm probability of one Bernoulli check at every cell size the GPU tests use, down to n = E / 256 at
  r = 0.001: at most ALPHA.
"""
import itertools

import numpy as np
import pytest

import control_oracle as CO
import law_oracle as L
from helpers import make_network, oracle_net
from oracle import pbn_oracle as O

E = 1 << 22


def _onet(n, kmax, amax, seed, uniform=False):
    return O.OracleNetwork(*make_network(n, kmax, amax, seed=seed, uniform=uniform))


def _enumerated_row(onet, s, flips, mode, p):
    """The law of the next state by pushing every (sel, pert) pair through O.batched_step."""
    n = onet.n
    sels = np.array(list(itertools.product(*[range(len(ps)) for ps in onet.probs])), dtype=np.uint8)
    psel = np.array([np.prod([onet.probs[i][k] for i, k in enumerate(row)]) for row in sels])
    masks = np.arange(1 << n, dtype=np.uint64) if (O.PERT_MODES[mode] and p > 0) else np.zeros(1, dtype=np.uint64)
    pm = CO.mask_probabilities(n, p) if masks.size > 1 else np.ones(1)
    sel = np.repeat(sels, masks.size, axis=0)
    pert = np.tile(masks, len(sels)).reshape(-1, 1)
    w = np.repeat(psel, masks.size) * np.tile(pm, len(sels))
    e = sel.shape[0]
    acts = np.zeros((e, 3), dtype=np.uint8)
    for j, g in enumerate([g for g in range(n) if (flips >> g) & 1][:3]):
        acts[:, j] = g + 1
    tables = O.attractor_tables([[tuple([0] * n)]], n)
    nxt = O.batched_step(onet, tables, np.full((e, 1), s, dtype=np.uint64), acts, np.zeros(e, np.int32),
                         np.zeros(e, np.uint16), horizon=0, mode=O.PERT_MODES[mode], sel=sel, pert=pert,
                         r_success=0.0, r_step=0.0, r_action=0.0)[0]
    out = np.zeros(1 << n)
    np.add.at(out, nxt[:, 0].astype(np.int64), w)
    return out


@pytest.mark.parametrize("mode,p", [("none", 0.0), ("A", 0.1), ("B", 0.1), ("C", 0.1), ("A", 0.6), ("C", 0.6)])
@pytest.mark.parametrize("seed", [5, 6])
def test_rows_against_enumeration(seed, mode, p):
    onet = _onet(5, 3, 3, seed)
    rng = np.random.default_rng(seed)
    for s in [0, 31] + [int(x) for x in rng.integers(0, 32, size=3)]:
        for flips in (0, 1 << int(rng.integers(5)), 0b10110):
            want = _enumerated_row(onet, s, flips, mode, p)
            got = L.projection(onet, s, flips, mode, p, list(range(5)))
            assert np.abs(got - want).max() <= 1e-13, (s, flips)
            marg = np.array([want[(np.arange(32) >> i) & 1 == 1].sum() for i in range(5)])
            assert np.abs(L.marginals(onet, s, flips, mode, p) - marg).max() <= 1e-13
            genes, law, fixed = L.full_row(onet, s, flips, mode, p)
            assert abs(law.sum() - 1.0) <= 1e-13
            for b, v in enumerate(law):
                t = fixed | sum(((b >> j) & 1) << g for j, g in enumerate(genes))
                assert abs(v - want[t]) <= 1e-13


@pytest.mark.parametrize("mode,p", [("none", 0.0), ("A", 0.05), ("B", 0.05), ("A", 0.5)])
@pytest.mark.parametrize("which", ["pbn7", "net8"])
def test_dense_against_transition_matrix(which, mode, p):
    onet = oracle_net("pbn7") if which == "pbn7" else _onet(8, 4, 3, seed=8)
    want = CO.transition_matrix(onet, mode, p)
    got = L.dense_matrix(onet, mode, p)
    assert np.abs(got - want).max() <= 1e-13


@pytest.mark.parametrize("mode,p", [("none", 0.0), ("A", 0.03), ("A", 0.3), ("B", 0.03), ("C", 0.2)])
def test_projection_against_full_row(mode, p):
    onet = _onet(11, 4, 3, seed=11)
    rng = np.random.default_rng(11)
    states = np.arange(1 << 11)
    for s in [0, 2047] + [int(x) for x in rng.integers(0, 2048, size=4)]:
        flips = int(rng.integers(0, 2048))
        full = L.projection(onet, s, flips, mode, p, list(range(11)))
        assert abs(full.sum() - 1.0) <= 1e-12
        for k in (1, 3, 7, 11):
            genes = [int(g) for g in rng.permutation(11)[:k]]
            idx = np.zeros(states.size, dtype=np.int64)
            for j, g in enumerate(genes):
                idx |= ((states >> g) & 1) << j
            want = np.bincount(idx, weights=full, minlength=1 << k)
            assert np.abs(L.projection(onet, s, flips, mode, p, genes) - want).max() <= 1e-13


def test_gene_probabilities():
    """q_i(s) from Python eval, from the numpy form and from control_oracle (which stops at 63 genes) agree; at 128
    genes the Python form and the numpy form agree and the probe network reads its probabilities back."""
    onet = _onet(40, 5, 4, seed=40)
    rng = np.random.default_rng(40)
    states = [int(x) for x in rng.integers(0, 1 << 40, size=64)]
    q = np.array([L.q_genes(onet, s) for s in states])
    assert np.abs(q - CO.gene_probabilities(onet, states)).max() <= 1e-15
    assert np.abs(q - L.q_states(onet, states)).max() <= 1e-15
    big = _onet(128, 4, 4, seed=128)
    states = [int(rng.integers(0, 1 << 62)) << 66 | int(rng.integers(0, 1 << 62)) for _ in range(16)]
    assert np.abs(np.array([L.q_genes(big, s) for s in states]) - L.q_states(big, states)).max() <= 1e-15
    layout = [None] * 4 + [[0.3, 0.2, 0.5], [0.999, 0.001], None, [1, 1, 1, 1]] + [None] * 60 + [[0.1, 0.9]]
    probe = O.OracleNetwork(*L.probe_network(layout, 4))
    law = L.probe_law(layout, 4)
    for j in range(4):
        assert np.abs(L.q_genes(probe, 1 << j) - law[j]).max() <= 1e-15
    # keep / negate networks: the step law is the mask law
    keep = O.OracleNetwork(*L.keep_network(6))
    for mode in ("A", "B", "C"):
        assert np.abs(L.projection(keep, 0, 0, mode, 0.2, range(6)) - L.product_law([0.2] * 6)).max() <= 1e-15
    neg = O.OracleNetwork(*L.negate_network(6))
    row = _enumerated_row(neg, 0b101100, 0, "A", 0.2)
    pc = np.array([bin(t ^ 0b101100).count("1") for t in range(64)])
    assert np.abs(np.bincount(pc, weights=row, minlength=7) - L.negate_flip_law(6, 0.2)).max() <= 1e-15


def test_reset_law():
    attrs = [[(0, 1, "*")], [(1, 1, 0), (0, 0, 1)], [(1, "*", "*"), (0, 1, 1), (1, 0, 1)]]
    law = L.reset_law(attrs)
    assert abs(law.sum() - 1.0) <= 1e-15
    assert law[0, 0].sum() == 0 and abs(law[2, 0, 0] - 1 / 18) <= 1e-15 and law[0, 1, 1] == 0
    assert L.reset_entries(attrs) == [[2], [3, 4], [1, 6, 5]]
    w = np.array([[0, 1, 0], [2, 0, 0], [0, 0, 1]], dtype=float)
    pl = L.reset_pair_law(3, w)
    assert pl.tolist() == [0, 0.25, 0, 0.5, 0, 0, 0, 0, 0.25]


# ---------------------------------------------------------------------------------------------- calibration
PROBE = [0.3, 0.2, 0.5]


def _probe_counts(rng, probs, per_code):
    """Counts of a probe gene over one-hot code states, as the GPU tests count them."""
    return np.array([rng.binomial(per_code, v) for v in probs])


@pytest.mark.parametrize("codes", [4, 8, 16])
def test_calibration_selection(codes):
    """Probe genes at the GPU split (E / codes envs per code state): the exact law passes the binomial rule; a probe
    whose probability is 2^-7 off fails it; the 12-gene joint law passes its chi-square."""
    rng = np.random.default_rng(codes)
    per = E // codes
    for probs in (PROBE, [0.5, 0.5], [0.999, 0.001], [0.25] * 4):
        j = L.Judge("exact")
        for _ in range(20):
            j.z(_probe_counts(rng, probs, per), per, probs, "exact")
        assert not j.failures, j.failures
        shifted = list(probs)
        k = int(np.argmax(shifted))
        shifted[k] -= 2.0 ** -7
        shifted[(k + 1) % len(shifted)] += 2.0 ** -7
        bad = L.Judge("shifted")
        bad.z(_probe_counts(rng, shifted, per), per, probs, "shifted")
        assert bad.failures and bad.max_z > 7.0, bad.report()
    joint = L.product_law([0.3, 0.2, 0.5, 0.5, 1 / 3, 1 / 3, 0.25, 0.999, 0.001, 0.7, 0.125, 0.6])
    j = L.Judge("joint")
    for _ in range(5):
        j.chi2((rng.multinomial(per, joint), joint), "joint")
    assert not j.failures, j.failures


@pytest.mark.parametrize("n,r", [(E // 256, 0.001), (E // 256, 0.0008), (E // 256, 0.999), (E // 256, 0.5),
                                 (E // 32, 1e-3), (E // 32, 0.9), (E // 16, 0.001), (E, 1e-3), (E // 4, 0.3)])
def test_calibration_binomial_size(n, r):
    """The exact false-alarm probability of one Bernoulli check at the GPU cell sizes -- down to a slice-bit cell of a
    rare predictor (n = E / 256 envs: 8 code blocks x 32 slice bits, r = 0.001, a mean of 16) -- summed over every
    count the rule rejects, is at most ALPHA.  The Gaussian rule |z| > 6 is far above it at the small means."""
    from scipy.stats import binom
    sd = np.sqrt(n * r * (1.0 - r))
    k = np.arange(max(0, int(n * r - 60 * sd) - 60), min(n, int(n * r + 60 * sd) + 60) + 1)
    pmf = binom.pmf(k, n, r)
    assert pmf.sum() > 1.0 - 1e-12
    size = float(pmf[L.binomial_p(k, n, r) < L.ALPHA].sum())
    assert size <= L.ALPHA, size
    gauss = float(pmf[np.abs(L.z_scores(k, n, r)) > L.Z_MAX].sum())
    if n * r < 20:
        assert gauss > 10 * L.ALPHA, gauss


def test_calibration_perturbation():
    """Keep network masks at E = 2^22: Binomial(N, p) popcounts and Bernoulli(p) genes pass; p * 1.05 fails both."""
    rng = np.random.default_rng(5)
    for n, p in ((28, 0.03), (64, 0.03), (128, 0.25), (1, 0.03)):
        for scale, passes in ((1.0, True), (1.05, False)):
            j = L.Judge("p x %.2f" % scale)
            pc = rng.multinomial(E, L.binomial_pmf(n, p * scale))
            j.chi2((pc, L.binomial_pmf(n, p)), "popcount")
            j.z(rng.binomial(E, p * scale, size=n), E, p, "genes")
            if passes:
                assert not j.failures, j.failures
            elif n > 1:
                assert j.min_p < 1e-12 and j.max_z > 6.0, j.report()
            else:                   # one gene: its total alone must catch the shift
                assert j.failures and j.max_z > 6.0, j.report()


def test_calibration_reused_selections():
    """A two-step law built as if step 2 reused step 1's selections is rejected against the exact two-step row; a
    sample of the exact row passes."""
    onet = _onet(5, 3, 3, seed=51)
    P = L.dense_matrix(onet, "none", 0.0)
    rng = np.random.default_rng(51)
    sels = list(itertools.product(*[range(len(ps)) for ps in onet.probs]))
    for s in (0, 13, 31):
        exact = (P @ P)[s]
        reused = np.zeros(32)
        for sel in sels:
            w = np.prod([onet.probs[i][k] for i, k in enumerate(sel)])
            t = onet.transition(onet.transition(s, 0, sel, 0, O.PERT_NONE), 0, sel, 0, O.PERT_NONE)
            reused[t] += w
        assert np.abs(reused - exact).sum() > 0.05
        good, bad = L.Judge("exact"), L.Judge("reused")
        good.chi2((rng.multinomial(E, exact), exact), "exact")
        bad.chi2((rng.multinomial(E, reused), exact), "reused")
        assert not good.failures and bad.failures, (good.report(), bad.report())


def test_decision_rule_edges():
    """A count where the probability is 0 fails at once; a certain outcome with a miss is an infinite z."""
    j = L.Judge("edges")
    j.chi2((np.array([10, 0, 1]), np.array([0.5, 0.5, 0.0])), "impossible")
    j.z(np.array([5]), 5, 0.0, "never")
    assert len(j.failures) == 2 and j.min_p == 0.0 and j.max_z == np.inf
    ok = L.Judge("edges ok")
    ok.z(np.array([0, 7]), 7, np.array([0.0, 1.0]), "certain")
    ok.chi2((np.array([7, 0]), np.array([1.0, 0.0])), "certain")
    assert not ok.failures
