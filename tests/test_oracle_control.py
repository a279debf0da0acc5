"""CPU: the dense restatement of exact finite-horizon control (tests/control_oracle.py) against the step contract
(oracle/pbn_oracle.py: batched_step), the ball relaxation of pbn_dp_improve against brute force, and the Bittner-7
optimum of the model_tester step count."""
import itertools

import numpy as np
import pytest

import control_oracle as CO
from helpers import golden, make_network, oracle_net
from oracle import pbn_oracle as O


def _net5():
    genes, exprs = make_network(5, 3, 3, seed=55, uniform=False)
    for row in exprs:   # three predictors per gene
        while len(row) < 3:
            row.append(row[0])
    tot = [sum(p for _, p in row) for row in exprs]
    exprs = [[(e, p / t) for e, p in row] for row, t in zip(exprs, tot)]
    return O.OracleNetwork(genes, exprs)


@pytest.mark.parametrize("mode", ["none", "A", "B"])
def test_transition_matrix_equals_enumerated_steps(mode):
    """P of the oracle = every (selection, perturbation mask) pair stepped through batched_step, weighted by its
    probability: the DP is pinned to the step contract."""
    onet = _net5()
    n, S, p = onet.n, 1 << onet.n, 0.07
    P = CO.transition_matrix(onet, mode, p)
    ref = np.zeros((S, S))
    sels = list(itertools.product(*[range(len(onet.probs[i])) for i in range(n)]))
    pm = CO.mask_probabilities(n, p) if mode != "none" else np.eye(1, S)[0]
    tables = O.attractor_tables([[tuple([0] * n)]], n)
    states = np.arange(S, dtype=np.uint64)
    for sel in sels:
        psel = float(np.prod([onet.probs[i][sel[i]] for i in range(n)]))
        for m in range(S):
            if pm[m] == 0.0:
                continue
            nxt, *_ = O.batched_step(onet, tables, states.reshape(-1, 1), np.zeros((S, 1), np.uint8),
                                     np.zeros(S, np.int32), np.zeros(S, np.uint16), horizon=0, mode=CO.MODES[mode],
                                     sel=np.tile(np.array(sel, np.uint8), (S, 1)),
                                     pert=np.full((S, 1), m, np.uint64), r_success=0.0, r_step=0.0, r_action=0.0)
            np.add.at(ref, (np.arange(S), nxt[:, 0].astype(np.int64)), psel * pm[m])
    assert np.abs(P - ref).max() < 1e-14
    assert np.abs(P.sum(axis=1) - 1.0).max() < 1e-14
    u = np.random.default_rng(1).standard_normal(S)
    assert np.abs(CO.expect(onet, u, mode, p) - P @ u).max() < 1e-13


def test_rows_match_exact_next_distribution():
    """At p = 0 every row of P is the exact next-state distribution of the perturbation-free update."""
    from test_gpu_env_api import _exact_next_distribution
    from helpers import product_net
    net, onet = product_net("pbn7"), oracle_net("pbn7")
    P = CO.transition_matrix(onet, "A", 0.0)
    for u in range(1 << 7):
        row = np.zeros(1 << 7)
        for t, pr in _exact_next_distribution(net, u).items():
            row[t] = pr
        assert np.abs(P[u] - row).max() < 1e-14
    big = CO.transition_matrix(onet, "A", 0.01)
    assert np.abs(big.sum(axis=1) - 1.0).max() < 1e-14


def _bittner7_matrix(mode, p):
    onet = oracle_net("pbn7")
    attrs = [[tuple(s) for s in a] for a in golden("attractors_bittner7.json")["attractors"]]
    P = CO.transition_matrix(onet, mode, p)
    a = len(attrs)
    reps = [O.bits_to_int(at[0]) for at in attrs]
    m = np.zeros((a, a))
    for t in range(a):
        hit, wrong = CO.classify(7, attrs, t)
        values, _ = CO.solve(P, hit, wrong, 100, (1 << 7) - 1, 3)
        m[:, t] = -values[100][reps]
    return m, attrs, reps


def test_bittner7_steps_optimum():
    """Bittner-7, bins = 3, perturbation off: the optimal policy's expected model_tester step count."""
    m, attrs, reps = _bittner7_matrix("none", 0.0)
    a = len(attrs)
    assert np.all(np.diag(m) == 0.0)
    for s in range(a):
        for t in range(a):
            if s == t:
                continue
            near = any(bin(reps[s] ^ O.bits_to_int(st)).count("1") <= 3 for st in attrs[t])
            if near:     # singleton attractors are closed (K2): one step lands in the target for sure
                assert m[s, t] == pytest.approx(1.0, abs=1e-12)
    off = m[~np.eye(a, dtype=bool)]
    assert off.mean() == pytest.approx(13.0 / 12.0, abs=1e-12)
    assert m[0, 1] == pytest.approx(4.0 / 3.0, abs=1e-12)
    assert m[0, 3] == pytest.approx(5.0 / 3.0, abs=1e-12)
    assert set(np.round(off, 12)) == {1.0, round(4.0 / 3.0, 12), round(5.0 / 3.0, 12)}


def test_bittner7_steps_optimum_model_a():
    m, attrs, _ = _bittner7_matrix("A", 0.01)
    off = m[~np.eye(len(attrs), dtype=bool)]
    assert np.all(np.diag(m) == 0.0)
    assert off.mean() == pytest.approx(1.1428279521589004, abs=1e-9)


@pytest.mark.parametrize("seed", range(6))
def test_ball_relaxation_equals_brute_force(seed):
    """The relaxation over one-flip neighbourhoods gives exactly the brute-force maximum and the contract's tie order,
    on values with deliberate ties and with ties created by rounding fl(r_action k) + w."""
    rng = np.random.default_rng(seed)
    n = int(rng.integers(3, 9))
    S = 1 << n
    kind = seed % 3
    if kind == 0:
        w = rng.integers(0, 4, size=S).astype(np.float64)            # many exact ties
        r_action = -1.0
    elif kind == 1:
        w = 1e16 + rng.integers(0, 3, size=S).astype(np.float64) * 2.0   # r_action * k is lost in the rounding
        r_action = -0.75
    else:
        w = rng.standard_normal(S)
        w[rng.integers(0, S, size=S // 3)] = w[0]
        r_action = float(rng.choice([0.0, -0.1, -1e-17]))
    for flip_genes in ((1 << n) - 1, int(rng.integers(0, 1 << n))):
        for max_flips in range(0, 6):
            vb, pb = CO.improve_brute(w, flip_genes, max_flips, r_action)
            vr, pr = CO.improve_ball(w, flip_genes, max_flips, r_action)
            assert np.array_equal(vb, vr)
            assert np.array_equal(pb, pr), (flip_genes, max_flips)


def test_three_gene_expectimax_equals_two_stage_dp():
    """Plain recursion over every action sequence of a 3-gene network (expectimax) = the 2-stage DP ("return")."""
    genes, exprs = make_network(3, 3, 2, seed=3, uniform=False)
    onet = O.OracleNetwork(genes, exprs)
    P = CO.transition_matrix(onet, "B", 0.05)
    attrs = [[(1, 0, 1)], [(0, "*", 0)]]
    hit, wrong = CO.classify(3, attrs, 0)
    kw = dict(r_success=5.0, r_step=-0.5, r_action=-1.0, r_wrong=-2.0, gamma=0.9)
    values, _ = CO.solve(P, hit, wrong, 2, 0b111, 2, objective="return", **kw)

    def rec(s, k):
        if k == 0:
            return 0.0
        best = -np.inf
        for m in CO.masks_of(0b111, 2):
            u = s ^ m
            q = kw["r_step"] + kw["r_action"] * bin(m).count("1")
            for t in range(8):
                r = kw["r_success"] if hit[t] else (kw["r_wrong"] if wrong[t] else 0.0)
                q += P[u, t] * (r + (0.0 if hit[t] else kw["gamma"] * rec(t, k - 1)))
            best = max(best, q)
        return best

    for s in range(8):
        assert values[2][s] == pytest.approx(rec(s, 2), abs=1e-12)
