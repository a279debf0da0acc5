"""CPU: the dense references of exact state distributions (tests/ssd_oracle.py) and the summaries of
pbn_rl_b200.steady_state.StateDistribution on host tensors."""
import numpy as np
import pytest

import control_oracle as CO
import ssd_oracle as SO
from helpers import make_network, oracle_net


def _net(n=6, seed=66):
    from oracle import pbn_oracle as O
    genes, exprs = make_network(n, 3, 3, seed=seed, uniform=False)
    return O.OracleNetwork(genes, exprs)


@pytest.mark.parametrize("mode,p", [("A", 0.01), ("A", 0.2), ("B", 0.01), ("B", 0.2)])
@pytest.mark.parametrize("name", ["net6", "pbn7"])
def test_stationary_solve_and_power_iteration(name, mode, p):
    onet = _net() if name == "net6" else oracle_net("pbn7")
    P = CO.transition_matrix(onet, mode, p)
    assert np.allclose(P.sum(axis=1), 1.0, atol=1e-14)
    pi = SO.stationary(P)
    assert np.all(pi > 0.0) and abs(pi.sum() - 1.0) <= 1e-14
    assert np.abs(pi @ P - pi).max() <= 1e-15
    x, it = SO.power_iteration(P, tol=1e-14)
    assert np.abs(x - pi).sum() <= 1e-10, it


@pytest.mark.parametrize("mode", ["none", "A", "B"])
def test_dense_transition_matches_the_enumeration(mode):
    """The product form used above 8 genes equals the row-by-row enumeration of control_oracle at 9 genes."""
    onet = _net(9, 99)
    assert onet.n == 9
    P = SO.dense_transition(onet, mode, 0.07)
    assert np.abs(P - CO.transition_matrix(onet, mode, 0.07)).max() <= 1e-15


def test_push_and_closed_loop():
    onet = _net()
    S = 1 << onet.n
    rng = np.random.default_rng(3)
    P = CO.transition_matrix(onet, "A", 0.05)
    x = rng.random(S)
    x /= x.sum()
    assert np.allclose(SO.push(onet, x, "A", 0.05, P=P), x @ P)
    masks = rng.integers(0, S, size=S)
    Pm = SO.closed_loop_matrix(onet, "A", 0.05, masks, P=P)
    M = np.zeros((S, S))
    M[np.arange(S), np.arange(S) ^ masks] = 1.0
    assert np.array_equal(Pm, M @ P)
    assert np.allclose(Pm.sum(axis=1), 1.0, atol=1e-14)
    assert np.array_equal(SO.closed_loop_matrix(onet, "A", 0.05, np.zeros(S, np.int64), P=P), P)


def test_point_row_matches_dense():
    onet = _net()
    F = CO.transition_matrix(onet)
    for s in range(1 << onet.n):
        t, w = SO.point_row(onet, s)
        row = np.zeros(1 << onet.n)
        row[t] = w
        assert np.abs(row - F[s]).max() <= 1e-15


def _hand_made():
    """4 genes: mass 0.5 on 0b0000, 0.25 on 0b0101, 0.125 on 0b1110 and 0b1011."""
    x = np.zeros(16)
    x[0b0000], x[0b0101], x[0b1110], x[0b1011] = 0.5, 0.25, 0.125, 0.125
    return x


def test_summaries_on_hand_made_vectors():
    import torch
    from pbn_rl_b200.steady_state import StateDistribution
    x = _hand_made()
    # gene 0: 0b0101, 0b1011; gene 1: 0b1110, 0b1011; gene 2: 0b0101, 0b1110; gene 3: 0b1110, 0b1011
    want_marg = np.array([0.375, 0.25, 0.375, 0.25])
    assert np.array_equal(SO.marginals(x), want_marg)
    d = StateDistribution(torch.from_numpy(x), 4)
    assert np.array_equal(d.marginals(), want_marg)
    # projection onto (gene 2, gene 0): bin bit 0 = gene 2, bit 1 = gene 0
    want = np.zeros(4)
    want[0b00] = 0.5            # 0b0000
    want[0b11] = 0.25           # 0b0101: gene 2 = 1, gene 0 = 1
    want[0b01] = 0.125          # 0b1110: gene 2 = 1, gene 0 = 0
    want[0b10] = 0.125          # 0b1011: gene 2 = 0, gene 0 = 1
    assert np.array_equal(SO.projection(x, [2, 0]), want)
    assert np.array_equal(d.projection([2, 0]), want)
    assert np.array_equal(d.projection([0, 1, 2, 3]), x)
    assert np.array_equal(d.projection([]), np.array([1.0]))
    assert d.mass([0b0101, 0b1011, 0b1011]) == 0.375
    assert d.mass(np.array([[0], [0b1110]], dtype=np.int64)) == 0.625
    with pytest.raises(ValueError):
        d.projection([1, 1])
    with pytest.raises(ValueError):
        d.projection([4])
    with pytest.raises(ValueError):
        d.mass([16])


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_summaries_on_random_vectors(seed):
    import torch
    from pbn_rl_b200.steady_state import StateDistribution
    rng = np.random.default_rng(seed)
    n = 7
    x = rng.random(1 << n)
    x /= x.sum()
    d = StateDistribution(torch.from_numpy(x), n)
    assert np.abs(d.marginals() - SO.marginals(x)).max() <= 1e-15
    for genes in ([3], [6, 0], [1, 5, 2], [4, 2, 0, 6, 1, 3, 5]):
        assert np.abs(d.projection(genes) - SO.projection(x, genes)).max() <= 1e-15, genes
