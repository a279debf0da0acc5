"""CPU: the dense restatement of exact finite-horizon control (tests/control_oracle.py) against the step contract
(oracle/pbn_oracle.py: batched_step), the ball relaxation of pbn_dp_improve against brute force, the Bittner-7
optimum of the model_tester step count, and the sampled references of the large-network tests against the dense
forms."""
import itertools

import numpy as np
import pytest

import control_oracle as CO
from helpers import golden, make_network, oracle_net, run_state, window_network
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


# ---- the references that scale to 2^28 states (tests/test_gpu_control_large.py) against the dense forms ------------
def _window_pair(n, k, seed):
    from pbn_rl_b200 import PBNNetwork
    genes, exprs = window_network(n, k, seed)
    return O.OracleNetwork(genes, exprs), PBNNetwork.from_expressions(genes, exprs)


def _window_terms(n, k):
    """sum_x 2^free(x) of window_network(n, k) as trace(T^n): T walks the windows of k consecutive genes, weight 2
    when the window it enters is all ones (the gene before that window is then free)."""
    t = np.zeros((1 << k, 1 << k), dtype=object)
    for a in range(1 << k):
        for bit in (0, 1):
            b = (a >> 1) | (bit << (k - 1))
            t[a, b] = 2 if b == (1 << k) - 1 else 1
    m = np.identity(1 << k, dtype=object)
    for _ in range(n):
        m = m.dot(t)
    return int(np.trace(m))


@pytest.mark.parametrize("n,k,seed", [(9, 3, 1), (10, 3, 2), (8, 6, 3)])
def test_window_network_free_counts(n, k, seed):
    """Gene i of window_network is free exactly when genes i+1..i+k (mod n) are all ones, in the oracle's expressions
    and in the product's truth tables; single runs and the all-ones state have the free counts the tests rely on, and
    the total successor count is the transfer-matrix trace."""
    onet, net = _window_pair(n, k, seed)
    s = np.arange(1 << n, dtype=np.int64)
    want = np.zeros(s.size, dtype=np.int64)
    for i in range(n):
        win = np.ones(s.size, dtype=bool)
        for j in range(1, k + 1):
            win &= ((s >> ((i + j) % n)) & 1).astype(bool)
        want += win
    assert np.array_equal(CO.free_counts(onet, s), want)
    assert np.array_equal(CO.free_counts(net, s), want)
    for start in range(n):
        for length in range(k, n):
            assert want[run_state(n, start, length)] == length - k + 1
        for length in range(k):
            assert want[run_state(n, start, length)] == 0
    assert want[(1 << n) - 1] == n
    assert int((np.ones(s.size, dtype=np.int64) << want).sum()) == _window_terms(n, k)
    assert all(np.array_equal(a, b) for a, b in zip(CO.gene_split(onet, s), CO.gene_split(net, s)))


def test_window_terms_at_the_sizes_of_the_large_tests():
    """The successor counts quoted for the large-N expect tests (sum_x 2^free(x))."""
    assert _window_terms(24, 3) == pytest.approx(1.5e9, rel=0.1)
    assert _window_terms(26, 3) == pytest.approx(9.1e9, rel=0.1)
    assert _window_terms(28, 3) == pytest.approx(5.4e10, rel=0.1)
    assert _window_terms(28, 6) == pytest.approx(2.0e9, rel=0.1)


@pytest.mark.parametrize("which", ["window", "random", "pbn10"])
def test_chunked_sparse_expect_equals_dense(which):
    """sparse_expect with the successor set cut into outer chunks (chunk_bits 0..3) and in one piece equals the dense
    F u, with u as an array and as a formula."""
    if which == "window":
        onet, _ = _window_pair(10, 3, 4)
    elif which == "random":
        genes, exprs = make_network(9, 3, 4, seed=9, uniform=False)
        onet = O.OracleNetwork(genes, exprs)
    else:
        onet = oracle_net("pbn10")
    n = onet.n
    s = np.arange(1 << n, dtype=np.int64)
    u = CO.u_hash(s)
    dense = CO.expect(onet, u)
    states = np.arange(0, 1 << n, 3)
    assert CO.free_counts(onet, states).max() >= 4
    ref = CO.sparse_expect(onet, u, states)
    assert np.abs(ref - dense[states]).max() <= 1e-14
    for cb in (0, 1, 3):
        assert np.abs(CO.sparse_expect(onet, CO.u_hash, states, chunk_bits=cb) - ref).max() <= 1e-15
    assert np.array_equal(CO.sparse_expect(onet, CO.u_hash, states), ref)


def test_formula_inputs_are_exact():
    """The formula inputs give the same fp64 values in numpy and torch, and u_hash is hash32 2^-32 - 0.5 exactly."""
    import torch
    t = np.concatenate([np.arange(1 << 12), (1 << 28) - 1 - np.arange(1 << 12), [1 << 27, 12345678]]).astype(np.int64)
    for f in (CO.u_hash, CO.w_ties, CO.w_rounding):
        a = f(t)
        b = f(torch.from_numpy(t)).numpy()
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64))
    h = np.array([(int(x) * 0x9E3779B1) % (1 << 32) for x in t])
    assert np.array_equal(CO.u_hash(t), np.array([float(v) / 2 ** 32 - 0.5 for v in h]))
    assert set(CO.w_ties(t)) == {0.0, 1.0, 2.0, 3.0}
    assert set(CO.w_rounding(t)) == {1e16, 1e16 + 2.0, 1e16 + 4.0}


@pytest.mark.parametrize("p", [1e-3, 0.05, 0.3])
def test_kp_tensor_equals_enumerated_masks(p):
    """K_p u as a tensor product of 2x2 channels equals the direct sum over every perturbation mask; with it the
    model A and model B references of the large tests equal the dense expect."""
    onet, _ = _window_pair(9, 3, 5)
    n = onet.n
    s = np.arange(1 << n, dtype=np.int64)
    u = CO.u_hash(s)
    kpu = CO.kp_tensor(u, p)
    assert np.abs(kpu - CO.kp_direct(u, s, p)).max() <= 1e-15
    states = s[::5]
    fu = CO.sparse_expect(onet, u, states)
    c = (1.0 - p) ** n
    model_a = c * fu + kpu[states] - c * u[states]
    assert np.abs(model_a - CO.expect(onet, u, "A", p)[states]).max() <= 1e-14
    model_b = CO.sparse_expect(onet, kpu, states)
    assert np.abs(model_b - CO.expect(onet, u, "B", p)[states]).max() <= 1e-14


@pytest.mark.parametrize("kind", ["ties", "rounding", "normal"])
def test_sampled_brute_force_equals_full(kind):
    """improve_brute_states at listed states equals improve_brute over all states, values bit for bit and policies,
    with w as an array and as a formula."""
    n = 10
    s = np.arange(1 << n, dtype=np.int64)
    f, r_action = {"ties": (CO.w_ties, -1.0), "rounding": (CO.w_rounding, -0.75), "normal": (CO.u_hash, -0.1)}[kind]
    w = f(s)
    states = np.random.default_rng(3).choice(1 << n, size=97, replace=False)
    for genes in ((1 << n) - 1, 0b1000100011, 0b0000010000):
        for kmax in range(0, 9):
            vb, pb = CO.improve_brute(w, genes, kmax, r_action)
            vs, ps = CO.improve_brute_states(w, states, genes, kmax, r_action)
            assert np.array_equal(vs, vb[states]) and np.array_equal(ps, pb[states]), (genes, kmax)
            vf, pf = CO.improve_brute_states(f, states, genes, kmax, r_action)
            assert np.array_equal(vf, vs) and np.array_equal(pf, ps)


def test_sampled_classify_equals_full():
    attrs = [[(1, 0, "*", 1, 0, 0, 1, 0)], [(0, "*", 0, 0, 1, "*", 1, 1), (1, 1, 1, 1, 0, 0, 0, 0)],
             [tuple([0] * 8)]]
    states = np.array([0, 1, 5, 77, 128, 200, 255, 0b01001101, 0b11110010, 0b00010110])
    for t in range(3):
        hit, wrong = CO.classify(8, attrs, t)
        hs, ws = CO.classify_states(8, attrs, t, states)
        assert np.array_equal(hs, hit[states]) and np.array_equal(ws, wrong[states])
        assert hit.any() and wrong.any()
