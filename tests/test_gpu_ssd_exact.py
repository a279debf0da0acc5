"""GPU: the exact forward operator pbn_dp_push and pbn_rl_b200/steady_state.py -- against the dense x P of
tests/ssd_oracle.py up to 12 genes, bit-identical from call to call (also across launch slices), dual to the verified
pbn_dp_expect at 20 and 24 genes, point-mass rows at 21 to 28 genes (Bittner-28 included) against the successor
enumeration, the stationary solver against the dense linear solve, exact against sampled statistics of the env, and
the refusals."""
import numpy as np
import pytest

import control_oracle as CO
import ssd_oracle as SO
from helpers import attractor_set, make_network, product_net, run_state, window_network

pytestmark = pytest.mark.gpu

PERT = [("none", 0.0), ("A", 0.0), ("A", 0.01), ("A", 0.2), ("B", 0.0), ("B", 0.01), ("B", 0.2)]


def _net(name):
    from pbn_rl_b200 import PBNNetwork
    if name in ("pbn7", "pbn10", "pbn28"):
        return product_net(name)
    if name == "net12":
        return PBNNetwork.from_expressions(*make_network(12, 3, 4, seed=12, uniform=False))
    if name == "net20":
        return PBNNetwork.from_expressions(*make_network(20, 3, 4, seed=20))
    if name == "net24":
        return PBNNetwork.from_expressions(*make_network(24, 2, 3, seed=24))
    raise KeyError(name)


def _env(net, mode="none", p=0.0, attractors=None, **kw):
    from pbn_rl_b200 import AttractorSet, VecPBNEnv
    n = net.n_genes
    if attractors is None:
        attractors = AttractorSet([[tuple([0] * n)]], n)
    kw.setdefault("kernel", "scalar")
    return VecPBNEnv(net, 1, attractors, device="cuda:0", perturb_mode="A" if mode == "none" else mode,
                     perturb_p=0.0 if mode == "none" else p, **kw)


def _bits(t):
    import torch
    return t.view(torch.int64)


def _release():
    import torch
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _inputs(S, rng):
    """A random distribution, a random sub-probability vector with zeros, and three point masses."""
    x = rng.random(S)
    sub = rng.random(S) * (rng.random(S) < 0.3)
    out = [x / x.sum(), 0.7 * sub / sub.sum()]
    for s in (0, S - 1, int(rng.integers(S))):
        e = np.zeros(S)
        e[s] = 1.0
        out.append(e)
    return out


# ---- 1. push against the dense x P ----------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,p", PERT)
@pytest.mark.parametrize("name", ["pbn7", "pbn10", "net12"])
def test_push_matches_dense(name, mode, p):
    import torch
    from pbn_rl_b200.control import _Backup
    net = _net(name)
    n, S = net.n_genes, 1 << net.n_genes
    P = SO.dense_transition(net, mode, p)
    env = _env(net, mode, p)
    bk = _Backup(env)
    rng = np.random.default_rng(n)
    flips = rng.integers(0, S, size=S)
    flips[rng.random(S) < 0.3] = 0
    for masks in (None, np.zeros(S, dtype=np.int64), flips):
        Pm = SO.closed_loop_matrix(net, mode, p, masks, P)
        m = None if masks is None else torch.from_numpy(masks).cuda()
        for j, x in enumerate(_inputs(S, rng)):
            xd = torch.from_numpy(x).cuda()
            y = bk.push(xd, m)
            want = x @ Pm
            err = np.abs(y.cpu().numpy() - want).max()
            assert err <= 1e-15, (masks is None, j, err)
            assert torch.equal(_bits(y), _bits(bk.push(xd, m)))
    env.close()


# ---- 2. determinism across launch slices ------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,p", [("none", 0.0), ("A", 0.01), ("B", 0.01)])
def test_push_deterministic_24(mode, p):
    """At 24 genes (four launches of 2^22 states) two calls give the same bits, with and without masks."""
    import torch
    from pbn_rl_b200.control import _Backup
    net = _net("net24")
    env = _env(net, mode, p)
    bk = _Backup(env)
    S = 1 << 24
    g = torch.Generator(device="cuda:0").manual_seed(24)
    x = torch.rand(S, dtype=torch.float64, device="cuda:0", generator=g)
    x /= x.sum()
    m = torch.randint(0, S, (S,), device="cuda:0", generator=g, dtype=torch.int64)
    for masks in (None, m):
        y = bk.push(x, masks)
        assert torch.equal(_bits(y), _bits(bk.push(x, masks)))
        assert abs(float(y.sum()) - 1.0) <= 1e-12
    del x, m, y
    bk = None
    env.close()
    _release()


# ---- 3. duality with expect at 20 and 24 genes ------------------------------------------------------------------------
@pytest.mark.parametrize("mode,p", [("none", 0.0), ("A", 0.01), ("B", 0.05)])
@pytest.mark.parametrize("name", ["net20", "net24"])
def test_push_dual_to_expect(name, mode, p):
    """<x P, u> = <x, P u>: the new operator against the one the control tests pin to the oracle, with and without
    masks (<x P_mu, u> = <x, (P u)[s ^ mu(s)]>)."""
    import torch
    from pbn_rl_b200.control import _Backup
    net = _net(name)
    env = _env(net, mode, p)
    bk = _Backup(env)
    S = 1 << net.n_genes
    g = torch.Generator(device="cuda:0").manual_seed(S)
    x = torch.rand(S, dtype=torch.float64, device="cuda:0", generator=g)
    x /= x.sum()
    u = CO.u_hash(torch.arange(S, dtype=torch.int64, device="cuda:0"))
    pu = bk.expect(u)
    m = torch.randint(0, S, (S,), device="cuda:0", generator=g, dtype=torch.int64)
    s = torch.arange(S, dtype=torch.int64, device="cuda:0")
    for masks, rhs in ((None, pu), (m, pu[s ^ m])):
        a = float((bk.push(x, masks) * u).sum())
        b = float((x * rhs).sum())
        assert abs(a - b) <= 1e-12 * float(u.abs().max()), (masks is None, a, b)
    del x, u, pu, m, s
    bk = None
    env.close()
    _release()


# ---- 4. point-mass rows at 21 to 28 genes -----------------------------------------------------------------------------
def _row_check(bk, net, s):
    import torch
    S = 1 << net.n_genes
    e = torch.zeros(S, dtype=torch.float64, device="cuda:0")
    e[s] = 1.0
    y = bk.push(e)
    t, w = SO.point_row(net, s)
    idx = torch.from_numpy(t).cuda()
    got = y[idx].cpu().numpy()
    assert np.abs(got - w).max() <= 1e-15, s
    y[idx] = 0.0
    assert not bool(y.any()), s          # nothing lands outside the successor set
    return t.size


@pytest.mark.parametrize("n", [21, 25])
def test_point_rows_window(n):
    """Window networks (tests/helpers.py): states with 0 to 22 free genes (up to five digit tables of the push
    kernel), in the first and the last launch."""
    from pbn_rl_b200 import PBNNetwork
    from pbn_rl_b200.control import _Backup
    net = PBNNetwork.from_expressions(*window_network(n, 3, n))
    env = _env(net)
    bk = _Backup(env)
    sizes = set()
    fs = (0, 1, 4, 5, 6, 9, 13, 17, 21) + ((22,) if n == 25 else ())
    for f in fs:
        length = f + 2 if f else 2
        for start in (0, n - length // 2):
            s = run_state(n, start, length)
            assert int(CO.free_counts(net, [s])[0]) == f
            sizes.add(_row_check(bk, net, s))
    assert max(sizes) == 1 << max(fs)
    bk = None
    env.close()
    _release()


def test_point_rows_bittner28():
    """Bittner-28: the state with the most free genes among 2^16 random ones (19), and states spread over the
    launches."""
    from pbn_rl_b200.control import _Backup
    net = product_net("pbn28")
    rng = np.random.default_rng(28)
    cand = rng.integers(0, 1 << 28, size=1 << 16)
    free = CO.free_counts(net, cand)
    top = int(cand[int(free.argmax())])
    states = [top, 0, (1 << 28) - 1] + [int(s) for s in rng.integers(0, 1 << 28, size=6)]
    env = _env(net, attractors=attractor_set("pbn28"))
    bk = _Backup(env)
    sizes = [_row_check(bk, net, s) for s in states]
    assert max(sizes) == 1 << 19, sizes
    bk = None
    env.close()
    _release()


# ---- 5. the stationary solver against the dense solve -----------------------------------------------------------------
@pytest.mark.parametrize("mode,p", [("A", 0.01), ("A", 0.1), ("B", 0.01), ("B", 0.1)])
@pytest.mark.parametrize("name", ["pbn7", "pbn10", "net12"])
def test_stationary_matches_dense(name, mode, p):
    from pbn_rl_b200 import stationary_distribution
    net = _net(name)
    pi = SO.stationary(SO.dense_transition(net, mode, p))
    env = _env(net, mode, p)
    d = stationary_distribution(env, tol=1e-13)
    assert d.converged and d.residual < 1e-13 and d.iterations >= 16
    got = d.probs.cpu().numpy()
    assert np.abs(got - pi).sum() <= 1e-9, (d.iterations, np.abs(got - pi).sum())
    assert np.abs(d.marginals() - SO.marginals(pi)).max() <= 1e-9      # bounded by the L1 error
    env.close()


def test_stationary_closed_loop_and_start():
    """Masks and an explicit start: against the dense stationary vector of M_mu P."""
    import torch
    from pbn_rl_b200 import stationary_distribution
    net = _net("pbn10")
    S = 1 << 10
    rng = np.random.default_rng(10)
    masks = np.where(rng.random(S) < 0.5, 0, 1 << rng.integers(0, 10, size=S))
    pi = SO.stationary(SO.closed_loop_matrix(net, "A", 0.05, masks))
    env = _env(net, "A", 0.05)
    for start in (None, 3, torch.tensor([[7]])):
        d = stationary_distribution(env, tol=1e-13, initial=start, masks=torch.from_numpy(masks))
        assert d.converged and np.abs(d.probs.cpu().numpy() - pi).sum() <= 1e-9
    env.close()


# ---- 6. exact against sampled statistics ------------------------------------------------------------------------------
def _chi_square_p(counts, probs, total):
    """p-value of observed ``counts`` against ``probs``, bins of expected count < 5 lumped into one; no count may
    fall where the probability is 0."""
    from scipy.stats import chisquare
    assert counts[probs == 0.0].sum() == 0
    exp = probs * total
    big = exp >= 5.0
    obs = np.append(counts[big], counts[~big].sum())
    ex = np.append(exp[big], exp[~big].sum())
    if ex[-1] == 0.0:
        obs, ex = obs[:-1], ex[:-1]
    ex *= obs.sum() / ex.sum()
    return float(chisquare(obs, ex).pvalue)


@pytest.mark.parametrize("name", ["pbn10", "net20"])
def test_exact_against_sampled(name):
    """steady_state_statistics over 2^20 envs after 300 steps of burn-in, one record per env (independent samples):
    marginals within 5 sigma of the exact ones, an 8-gene projection by chi-square."""
    import torch
    from pbn_rl_b200 import AttractorSet, VecPBNEnv, stationary_distribution
    from pbn_rl_b200.discover import steady_state_statistics
    net = _net(name)
    n = net.n_genes
    attrs = attractor_set(name) if name == "pbn10" else AttractorSet([[tuple([0] * n)]], n)
    genes = [n - 1, 0, 3, 7, 2, 5, 1, 6] if n > 8 else [9, 0, 3, 7, 2, 5, 1, 6]
    one = _env(net, "A", 0.05, attractors=attrs)
    exact = stationary_distribution(one, tol=1e-13)
    one.close()
    E = 1 << 20
    env = VecPBNEnv(net, E, attrs, device="cuda:0", perturb_p=0.05, perturb_mode="A", horizon=0, seed=2024)
    env.set_state(torch.randint(0, 1 << n, (E, 1), dtype=torch.int64), packed=True)
    rec = steady_state_statistics(env, steps=1, burn_in=300, genes=genes)
    m_exact = exact.marginals()
    sigma = np.sqrt(m_exact * (1.0 - m_exact) / E)
    assert np.all(np.abs(rec.marginals() - m_exact) <= 5 * sigma + 1e-12), (rec.marginals(), m_exact)
    counts = rec.counts()[1].astype(np.float64)
    assert counts.sum() == E
    assert _chi_square_p(counts, exact.projection(genes), E) > 1e-6
    env.close()


# ---- 7. transient distributions -------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,p", [("none", 0.0), ("A", 0.05), ("B", 0.05)])
def test_transient_against_rollout(mode, p):
    """propagate(start, k) for k = 1..5 against 2^20 envs run k steps from the same start, recorded over all ten
    genes of Bittner-10, by chi-square."""
    import torch
    from pbn_rl_b200 import VecPBNEnv, propagate
    from pbn_rl_b200.discover import StateRecorder
    net, attrs = product_net("pbn10"), attractor_set("pbn10")
    start = 0b1011001110
    one = _env(net, mode, p, attractors=attrs)
    dists = propagate(one, start, 5, keep=True)
    one.close()
    assert len(dists) == 6 and float(dists[0].probs[start]) == 1.0
    E = 1 << 20
    env = VecPBNEnv(net, E, attrs, device="cuda:0", perturb_p=p, perturb_mode="A" if mode == "none" else mode,
                    horizon=0, seed=77)
    env.set_state(torch.full((E, 1), start, dtype=torch.int64), packed=True)
    genes = list(range(10))
    for k in range(1, 6):
        env.rollout(1, stats=False)
        rec = StateRecorder(env, genes=genes, marginals=False)
        rec.add()
        counts = rec.counts()[1].astype(np.float64)
        assert _chi_square_p(counts, dists[k].probs.cpu().numpy(), E) > 1e-6, k
        assert np.abs(dists[k].projection(genes) - dists[k].probs.cpu().numpy()).max() == 0.0
    env.close()


def test_propagate_closed_loop_matches_dense():
    import torch
    from pbn_rl_b200 import propagate
    net = _net("pbn7")
    rng = np.random.default_rng(7)
    masks = rng.integers(0, 128, size=128)
    Pm = SO.closed_loop_matrix(net, "B", 0.02, masks)
    env = _env(net, "B", 0.02)
    x = np.zeros(128)
    x[5] = 1.0
    d = propagate(env, 5, 4, masks=torch.from_numpy(masks))
    for _ in range(4):
        x = x @ Pm
    assert d.steps == 4 and np.abs(d.probs.cpu().numpy() - x).max() <= 1e-15
    assert propagate(env, x, 0).probs.cpu().numpy().tolist() == x.tolist()
    env.close()


# ---- 8. refusals ------------------------------------------------------------------------------------------------------
def test_refusals():
    import torch
    from pbn_rl_b200 import AttractorSet, PBNNetwork, VecPBNEnv, propagate, stationary_distribution
    from pbn_rl_b200._cabi import PBN_ERR_INVALID, PBN_ERR_UNSUPPORTED, PbnError
    from pbn_rl_b200.control import _Backup
    genes, exprs = make_network(29, 1, 2, seed=29)
    big = VecPBNEnv(PBNNetwork.from_expressions(genes, exprs), 1, AttractorSet([[tuple([0] * 29)]], 29), device="cuda:0",
                    kernel="scalar")
    lib = big.lib
    x = torch.zeros(4, dtype=torch.float64, device="cuda:0")
    assert lib.pbn_dp_push(big._h, x.data_ptr(), x.data_ptr(), None, x[2:].data_ptr(), None, None) == PBN_ERR_UNSUPPORTED
    with pytest.raises(PbnError):
        propagate(big, 0, 1)
    big.close()
    net = _net("pbn7")
    cenv = _env(net, "C", 0.01)
    assert lib.pbn_dp_push(cenv._h, x.data_ptr(), x.data_ptr(), None, x[2:].data_ptr(), None, None) == PBN_ERR_UNSUPPORTED
    with pytest.raises(PbnError):
        stationary_distribution(cenv)
    cenv.close()
    env = _env(net, "A", 0.01)
    bk = _Backup(env)
    fp, ws, h = bk.func_prob.data_ptr(), bk.ws.data_ptr(), env._h
    a = torch.zeros(128, dtype=torch.float64, device="cuda:0")
    a[0] = 1.0
    y = torch.zeros_like(a)
    m = torch.zeros(128, dtype=torch.int32, device="cuda:0")
    assert lib.pbn_dp_push(h, None, a.data_ptr(), None, y.data_ptr(), ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_push(h, fp, None, None, y.data_ptr(), ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_push(h, fp, a.data_ptr(), None, None, ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_push(h, fp, a.data_ptr(), None, a.data_ptr(), ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_push(h, fp, a.data_ptr(), None, y.data_ptr(), None, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_push(h, fp, a.data_ptr(), m.data_ptr(), y.data_ptr(), ws, None) == 0
    env.close()
    e0 = _env(net)
    b0 = _Backup(e0)
    assert lib.pbn_dp_push(e0._h, b0.func_prob.data_ptr(), a.data_ptr(), None, y.data_ptr(), None, None) == 0
    assert lib.pbn_dp_push(e0._h, b0.func_prob.data_ptr(), a.data_ptr(), m.data_ptr(), y.data_ptr(), None,
                           None) == PBN_ERR_INVALID      # masks need the workspace even at p = 0
    torch.cuda.synchronize()
    neg = torch.full((128,), 1.0 / 128, dtype=torch.float64)
    neg[3] = -1e-3
    with pytest.raises(ValueError):
        propagate(e0, neg, 1)
    with pytest.raises(ValueError):
        propagate(e0, torch.full((128,), 1.0 / 127, dtype=torch.float64), 1)
    with pytest.raises(ValueError):
        propagate(e0, 0, 1, masks=torch.full((128,), 1 << 7, dtype=torch.int64))
    with pytest.raises(ValueError):
        propagate(e0, 128, 1)
    with pytest.raises(ValueError):
        stationary_distribution(e0)
    assert propagate(e0, torch.full((128,), 1.0 / 128, dtype=torch.float64), 1).probs.sum().item() == pytest.approx(1.0)
    e0.close()
