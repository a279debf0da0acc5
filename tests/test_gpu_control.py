"""GPU: exact finite-horizon control (pbn_dp_expect / pbn_dp_improve, pbn_rl_b200/control.py) against the dense
oracle (tests/control_oracle.py), bit-exactness and determinism of the maximisation, the refusals, and end-to-end
agreement of the optimal policy's Monte Carlo scores with its exact values."""
import json

import numpy as np
import pytest

import control_oracle as CO
from helpers import GOLD, attractor_set, make_network, product_net

pytestmark = pytest.mark.gpu

PERT = [("none", 0.0), ("A", 1e-3), ("A", 0.05), ("B", 1e-3), ("B", 0.05)]


def _net(name):
    from pbn_rl_b200 import PBNNetwork
    if name in ("pbn7", "pbn10"):
        return product_net(name)
    if name == "control14":
        d = json.loads((GOLD / "control14.json").read_text())
        return PBNNetwork.from_logic_functions(d["genes"], d["logic_functions"])
    spec = {"syn1": (1, 3, 1, 11), "syn2": (2, 4, 2, 12), "syn12_weighted8": (12, 8, 3, 13),
            "syn10_wide": (10, 3, 9, 14)}[name]
    genes, exprs = make_network(spec[0], spec[1], spec[2], seed=spec[3], uniform=False)
    return PBNNetwork.from_expressions(genes, exprs)


def _env(net, mode="A", p=0.0, attractors=None, **kw):
    """A one-env handle for the backups (the general step kernel: nothing is stepped, no specialisation is built)."""
    from pbn_rl_b200 import VecPBNEnv, find_attractors_stg
    if attractors is None:
        attractors = find_attractors_stg(net)[0]
    kw.setdefault("kernel", "scalar")
    return VecPBNEnv(net, 1, attractors, device="cuda:0", perturb_mode=mode if mode != "none" else "A",
                     perturb_p=p if mode != "none" else 0.0, **kw)


@pytest.mark.parametrize("mode,p", PERT)
@pytest.mark.parametrize("name", ["pbn7", "pbn10", "control14", "syn1", "syn2", "syn12_weighted8", "syn10_wide"])
def test_expect_matches_oracle(name, mode, p):
    import torch
    from pbn_rl_b200.control import _Backup
    net = _net(name)
    env = _env(net, mode, p)
    bk = _Backup(env)
    rng = np.random.default_rng(len(name))
    u = rng.standard_normal(1 << net.n_genes) * 3.0
    got = bk.expect(torch.from_numpy(u).cuda()).cpu().numpy()
    want = CO.expect(net, u, mode, p)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(u).max()
    again = bk.expect(torch.from_numpy(u).cuda()).cpu().numpy()
    assert np.array_equal(got.view(np.uint64), again.view(np.uint64))     # deterministic
    env.close()


@pytest.mark.parametrize("n,kmax,amax,seed", [(16, 3, 4, 16), (20, 3, 4, 20)])
def test_expect_sparse_oracle_large(n, kmax, amax, seed):
    """Networks of 16 and 20 genes at p = 0: a sample of states against successor-set enumeration."""
    import torch
    from pbn_rl_b200 import AttractorSet, PBNNetwork
    from pbn_rl_b200.control import _Backup
    genes, exprs = make_network(n, kmax, amax, seed=seed)
    net = PBNNetwork.from_expressions(genes, exprs)
    env = _env(net, "none", 0.0, attractors=AttractorSet([[tuple([0] * n)]], n))
    bk = _Backup(env)
    rng = np.random.default_rng(seed)
    u = rng.standard_normal(1 << n)
    got = bk.expect(torch.from_numpy(u).cuda()).cpu().numpy()
    states = rng.choice(1 << n, size=120, replace=False)
    want = CO.sparse_expect(net, u, states)
    assert np.abs(got[states] - want).max() <= 1e-12 * np.abs(u).max()
    again = bk.expect(torch.from_numpy(u).cuda()).cpu().numpy()
    assert np.array_equal(got.view(np.uint64), again.view(np.uint64))
    env.close()


def _improve(bk, w, genes, kmax, r_action):
    import torch
    v, pol = bk.improve(torch.from_numpy(w).cuda(), genes, kmax, r_action)
    return v.cpu().numpy(), pol.cpu().numpy().astype(np.int64)


@pytest.mark.parametrize("kind", ["ties", "rounding", "normal", "backup"])
def test_improve_bit_identical_to_brute_force(kind):
    import torch
    from pbn_rl_b200.control import _Backup
    net = _net("pbn10")
    env = _env(net, "A", 0.01)
    bk = _Backup(env)
    rng = np.random.default_rng(7)
    S = 1 << 10
    if kind == "ties":
        w, r_action = rng.integers(0, 4, size=S).astype(np.float64), -1.0
    elif kind == "rounding":
        w, r_action = 1e16 + 2.0 * rng.integers(0, 3, size=S).astype(np.float64), -0.75
    elif kind == "normal":
        w, r_action = rng.standard_normal(S), -0.1
    else:
        w = bk.expect(torch.from_numpy(rng.standard_normal(S)).cuda()).cpu().numpy()
        r_action = -0.05
    for genes in ((1 << 10) - 1, 0b1011001101, 0b0000100000):
        for kmax in range(0, 9):
            vg, pg = _improve(bk, w, genes, kmax, r_action)
            vb, pb = CO.improve_brute(w, genes, kmax, r_action)
            assert np.array_equal(vg.view(np.uint64), vb.view(np.uint64)), (genes, kmax)
            assert np.array_equal(pg, pb), (genes, kmax)
            v2, p2 = _improve(bk, w, genes, kmax, r_action)
            assert np.array_equal(vg.view(np.uint64), v2.view(np.uint64)) and np.array_equal(pg, p2)
    env.close()


def test_refusals():
    import torch
    from pbn_rl_b200 import AttractorSet, PBNNetwork, VecPBNEnv
    from pbn_rl_b200._cabi import PBN_ERR_INVALID, PBN_ERR_UNSUPPORTED
    from pbn_rl_b200.control import _Backup
    genes, exprs = make_network(29, 1, 2, seed=29)
    big = VecPBNEnv(PBNNetwork.from_expressions(genes, exprs), 1, AttractorSet([[tuple([0] * 29)]], 29), device="cuda:0",
                    kernel="scalar")
    lib = big.lib
    assert lib.pbn_dp_workspace_bytes(big._h) == PBN_ERR_UNSUPPORTED
    x = torch.zeros(4, dtype=torch.float64, device="cuda:0")
    assert lib.pbn_dp_expect(big._h, x.data_ptr(), x.data_ptr(), x[2:].data_ptr(), None, None) == PBN_ERR_UNSUPPORTED
    assert lib.pbn_dp_improve(big._h, x.data_ptr(), 1, 1, -1.0, x[2:].data_ptr(), None, None, None) == PBN_ERR_UNSUPPORTED
    big.close()
    net = _net("pbn7")
    cenv = _env(net, "C", 0.01)
    assert lib.pbn_dp_workspace_bytes(cenv._h) == PBN_ERR_UNSUPPORTED
    assert lib.pbn_dp_expect(cenv._h, x.data_ptr(), x.data_ptr(), x[2:].data_ptr(), None, None) == PBN_ERR_UNSUPPORTED
    cenv.close()
    c0 = _env(net, "C", 0.0)     # model C without perturbation is NONE
    assert lib.pbn_dp_workspace_bytes(c0._h) == 24 * 128
    c0.close()
    env = _env(net, "A", 0.01)
    bk = _Backup(env)
    w = torch.zeros(128, dtype=torch.float64, device="cuda:0")
    v = torch.zeros_like(w)
    ws = bk.ws.data_ptr()
    h = env._h
    assert lib.pbn_dp_improve(h, w.data_ptr(), 0x7F, 3, 0.5, v.data_ptr(), None, ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_improve(h, w.data_ptr(), 0x7F, 9, -1.0, v.data_ptr(), None, ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_improve(h, w.data_ptr(), 0xFF, 3, -1.0, v.data_ptr(), None, ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_improve(h, None, 0x7F, 3, -1.0, v.data_ptr(), None, ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_improve(h, w.data_ptr(), 0x7F, 3, -1.0, None, None, ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_improve(h, w.data_ptr(), 0x7F, 3, -1.0, v.data_ptr(), None, None, None) == PBN_ERR_INVALID
    fp = bk.func_prob.data_ptr()
    assert lib.pbn_dp_expect(h, None, w.data_ptr(), v.data_ptr(), ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_expect(h, fp, None, v.data_ptr(), ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_expect(h, fp, w.data_ptr(), None, ws, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_expect(h, fp, w.data_ptr(), v.data_ptr(), None, None) == PBN_ERR_INVALID
    assert lib.pbn_dp_improve(h, w.data_ptr(), 0x7F, 3, -1.0, v.data_ptr(), None, ws, None) == 0
    env.close()


def _solutions(net, attrs, mode, p, stages=100):
    from pbn_rl_b200 import solve_control
    env = _env(net, mode, p, attractors=attrs, bins=3, horizon=0)
    sols = {t: solve_control(env, t, objective="steps", stages=stages) for t in range(len(attrs))}
    return env, sols


def _pair_samples(net, attrs, policy, runs, mode, p):
    import torch
    from pbn_rl_b200.evaluate import evaluate_all_pairs
    m, _, env, info = evaluate_all_pairs(net, attrs, policy, runs=runs, perturb_p=p, perturb_mode=mode if mode != "none" else "A",
                                         return_env=True)
    a = len(attrs)
    counts = info["count"].cpu().numpy().reshape(runs, a * a).astype(np.float64)
    env.close()
    return m, counts


@pytest.mark.parametrize("mode,p", [("none", 0.0), ("A", 0.01)])
@pytest.mark.parametrize("name", ["pbn7", "pbn10"])
def test_optimal_policy_all_pairs_monte_carlo(name, mode, p):
    """evaluate_all_pairs with the tabulated optimal policy: each pair's mean count within 5 sigma of the exact
    expectation."""
    from pbn_rl_b200 import TabularPolicy, expected_all_pairs
    net, attrs = product_net(name), attractor_set(name)
    env, sols = _solutions(net, attrs, mode, p)
    exact = expected_all_pairs(env, attrs, sols)
    runs = 4096
    m, counts = _pair_samples(net, attrs, TabularPolicy(sols), runs, mode, p)
    a = len(attrs)
    mean = counts.mean(axis=0).reshape(a, a)
    sem = counts.std(axis=0, ddof=1).reshape(a, a) / np.sqrt(runs)
    assert np.allclose(m / runs, mean)
    assert np.all(np.abs(mean - exact) <= 5 * sem + 1e-9), (mean, exact, sem)
    if name == "pbn7" and mode == "none":
        off = exact[~np.eye(a, dtype=bool)]
        assert off.mean() == pytest.approx(13.0 / 12.0, abs=1e-12)
    env.close()


def test_return_objective_rollouts():
    """VecPBNEnv rollouts of the "return" policy over a horizon of 20 from fixed start states: the mean return lies
    within 5 sigma of V_20."""
    import torch
    from pbn_rl_b200 import VecPBNEnv, solve_control
    net, attrs = product_net("pbn10"), attractor_set("pbn10")
    kw = dict(horizon=20, bins=3, perturb_p=0.01, perturb_mode="A", r_success=5.0, r_step=-0.25, r_action=-1.0,
              r_wrong=-2.0)
    solver = VecPBNEnv(net, 1, attrs, device="cuda:0", **kw)
    target = 0
    sol = solve_control(solver, target)
    starts = [0, 0b1010110011, 0b0111000101, 1023]
    per = 1 << 14
    e = per * len(starts)
    env = VecPBNEnv(net, e, attrs, device="cuda:0", seed=99, **kw)
    s0 = torch.tensor(starts, dtype=torch.int64, device="cuda:0").repeat_interleave(per)
    env.set_state(s0.unsqueeze(1), packed=True)
    env.set_target(torch.full((e,), target, dtype=torch.int32))
    env.t.zero_()
    ret = torch.zeros(e, dtype=torch.float64, device="cuda:0")
    active = torch.ones(e, dtype=torch.bool, device="cuda:0")
    for t in range(20):
        act = sol.actions(env.state, steps_left=20 - t)
        env.step(act)
        ret += torch.where(active, env.reward.to(torch.float64), 0.0)
        active &= ~(env.terminated.bool() | env.truncated.bool())
    assert not bool(active.any())
    r = ret.cpu().numpy().reshape(len(starts), per)
    v = sol.value(torch.tensor(starts), steps_left=20).cpu().numpy()
    sem = r.std(axis=1, ddof=1) / np.sqrt(per)
    assert np.all(np.abs(r.mean(axis=1) - v) <= 5 * sem + 1e-9), (r.mean(axis=1), v, sem)
    env.close()
    solver.close()


def test_policy_values_of_hamming_policy():
    """policy_values of a hand-written policy (tabulated over all states) matches its Monte Carlo all-pairs scores
    and never exceeds the optimum."""
    import torch
    from pbn_rl_b200 import policy_values, tabulate_policy
    from pbn_rl_b200.evaluate import hamming_policy
    net, attrs = product_net("pbn10"), attractor_set("pbn10")
    mode, p = "A", 0.01
    env, sols = _solutions(net, attrs, mode, p)
    a = len(attrs)
    reps = attrs.representative_words()[:, 0].astype(np.int64)
    exact = np.zeros((a, a))
    for t in range(a):
        masks = tabulate_policy(hamming_policy(3), env, t)
        pv = policy_values(env, t, masks, objective="steps", stages=100)
        assert bool((pv[100] <= sols[t].values[100] + 1e-9).all())
        exact[:, t] = -pv[100][torch.from_numpy(reps)].cpu().numpy()
    runs = 4096
    _, counts = _pair_samples(net, attrs, hamming_policy(3), runs, mode, p)
    mean = counts.mean(axis=0).reshape(a, a)
    sem = counts.std(axis=0, ddof=1).reshape(a, a) / np.sqrt(runs)
    assert np.all(np.abs(mean - exact) <= 5 * sem + 1e-9), (mean, exact, sem)
    env.close()


def test_control_env_flips_only_control_genes():
    from pbn_rl_b200 import ControlPBNEnv, solve_control
    d = json.loads((GOLD / "control14.json").read_text())
    env = ControlPBNEnv(genes=d["genes"], logic_functions=d["logic_functions"], control_nodes=d["control_nodes"],
                        horizon=10, perturb_p=0.01, kernel="scalar")
    allowed = sum(1 << c for c in d["control_nodes"] if c < 14)
    for t in range(len(env.all_attractors)):
        sol = solve_control(env, t)
        assert sol.flip_genes == allowed and sol.max_flips == 7
        pol = sol.policies.cpu().numpy().astype(np.int64)
        assert np.all((pol & ~allowed) == 0)
        assert (pol != 0).any()
    env.close()
