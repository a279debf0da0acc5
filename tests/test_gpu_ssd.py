"""GPU: steady-state statistics recorded on the device -- pbn_rollout_record (inside the rollout kernel) and
pbn_record_states (after a step) -- against the oracle's record contract (oracle/record_oracle.py) over the states the
oracle walks through the sliced random streams, against pbn_rollout, against steady_state_histogram and against the
exact Markov chain of Bittner-7."""
import ctypes as C

import numpy as np
import pytest

from helpers import attractor_set, oracle_net, product_net

pytestmark = pytest.mark.gpu

SIZES = {"pbn7": 33, "pbn10": 1024, "pbn28": 3000, "pbn70": 2053}
PROJ = {"pbn7": [6, 0, 3, 1, 5, 2, 4], "pbn10": [9, 2, 0, 7, 4, 1, 8, 3, 6, 5],
        "pbn28": [27, 3, 14, 0, 21, 8, 11, 25, 1, 17, 6, 12],
        "pbn70": [69, 3, 64, 12, 40, 0, 65, 31, 32, 63, 7, 50]}   # unsorted; pbn70: genes of both words
MODES = {"A": 1, "B": 2, "C": 3}


def _start(name, e):
    net = product_net(name)
    rng = np.random.default_rng(7)
    masks = np.array(net.state_mask(), dtype=np.uint64)
    return ((rng.integers(0, 2**63, size=(e, net.n_words), dtype=np.int64).astype(np.uint64) * np.uint64(2)
             + rng.integers(0, 2, size=(e, net.n_words)).astype(np.uint64)) & masks)


def _env(name, e, p, mode, st, **kw):
    import torch
    from pbn_rl_b200 import VecPBNEnv
    kw.setdefault("seed", 99)
    env = VecPBNEnv(product_net(name), e, attractor_set(name), device="cuda:0", perturb_p=p, perturb_mode=mode,
                    horizon=0, **kw)
    env.set_state(torch.from_numpy(st.astype(np.int64)), packed=True)
    return env


_TRAJ = {}


def _oracle_states(name, mode, p, n_steps=7):
    """States after updates 1..n_steps, walked by the oracle through the sliced streams."""
    key = (name, mode, p)
    if key not in _TRAJ:
        from oracle import pbn_oracle as O
        e = SIZES[name]
        onet = oracle_net(name)
        ids = np.arange(e, dtype=np.uint64)
        state = _start(name, e)
        zero = np.zeros((e, state.shape[1]), dtype=np.uint64)
        out = []
        for step in range(n_steps):
            sel, pert = O.sliced_stream(onet, p, ids, step, 99)
            state = onet.transition_batch(state, zero, sel, pert, MODES[mode])
            out.append(state.copy())
        _TRAJ[key] = out
    return _TRAJ[key]


def _oracle_counts(states, n, genes):
    from oracle.record_oracle import record_states
    on = np.zeros(n, dtype=np.uint64)
    hist = None if genes is None else np.zeros(1 << len(genes), dtype=np.uint64)
    for st in states:
        a, b = record_states(st, n, genes)
        on += a
        if hist is not None:
            hist += b
    return on, hist


@pytest.mark.parametrize("name", list(SIZES))
@pytest.mark.parametrize("mode,p", [("A", 0.0), ("A", 0.03), ("B", 0.03), ("C", 0.03)])
@pytest.mark.parametrize("stride", [1, 3])
def test_rollout_record_matches_the_oracle(name, mode, p, stride):
    from pbn_rl_b200.discover import StateRecorder
    e, n = SIZES[name], product_net(name).n_genes
    traj = _oracle_states(name, mode, p)
    recorded = [traj[s - 1] for s in range(1, 8) if s % stride == 0]
    for genes in ([], [n - 1], PROJ[name][:min(12, n)]):
        env = _env(name, e, p, mode, _start(name, e))
        rec = StateRecorder(env, genes=genes)
        env.rollout(7, recorder=rec, stride=stride)
        on, hist = rec.counts()
        ref_on, ref_hist = _oracle_counts(recorded, n, genes)
        assert np.array_equal(env.state.cpu().numpy().astype(np.uint64), traj[-1]), (name, genes)
        assert np.array_equal(on, ref_on), (name, mode, p, stride, genes)
        assert np.array_equal(hist, ref_hist), (name, mode, p, stride, genes)
        assert rec.n == e * len(recorded)
        env.close()


def test_rollout_record_leaves_the_rollout_unchanged():
    import torch
    from pbn_rl_b200.discover import StateRecorder
    name, e = "pbn28", (1 << 16) + 37
    st = _start(name, e)
    for p in (0.0, 0.01):
        ref, dut, loop = (_env(name, e, p, "A", st) for _ in range(3))
        rec = StateRecorder(dut, genes=PROJ[name][:8])
        ref_rec = StateRecorder(loop, genes=PROJ[name][:8])
        ref.rollout(64)
        dut.rollout(64, recorder=rec)
        for _ in range(64):
            loop.rollout(1)
            ref_rec.add()
        torch.cuda.synchronize()
        assert torch.equal(ref.state, dut.state) and torch.equal(ref.state, loop.state)
        assert ref.stats() == dut.stats()
        for a, b in zip(rec.counts(), ref_rec.counts()):
            assert np.array_equal(a, b)
        assert int(rec.counts()[1].sum()) == 64 * e
        for x in (ref, dut, loop):
            x.close()


def test_record_accumulates_accepts_null_and_shards():
    import torch
    from pbn_rl_b200.discover import StateRecorder
    name, e = "pbn28", 4096
    st = _start(name, e)
    genes = PROJ[name][:6]
    whole = _env(name, e, 0.02, "A", st)
    rec = StateRecorder(whole, genes=genes)
    whole.rollout(3, recorder=rec, stride=1)
    whole.rollout(4, recorder=rec, stride=2)          # two calls add up
    twin = _env(name, e, 0.02, "A", st)
    r1, r2 = StateRecorder(twin, genes=genes), StateRecorder(twin, genes=genes)
    twin.rollout(3, recorder=r1, stride=1)
    twin.rollout(4, recorder=r2, stride=2)
    for a, b, c in zip(rec.counts(), r1.counts(), r2.counts()):
        assert np.array_equal(a, b + c)
    assert rec.n == 5 * e
    # NULL gene_on / NULL hist
    only_hist = _env(name, e, 0.02, "A", st)
    only_on = _env(name, e, 0.02, "A", st)
    rh, ro = StateRecorder(only_hist, genes=genes, marginals=False), StateRecorder(only_on, genes=None)
    only_hist.rollout(3, recorder=rh)
    only_on.rollout(3, recorder=ro)
    assert rh.counts()[0] is None and ro.counts()[1] is None
    assert np.array_equal(rh.counts()[1], r1.counts()[1]) and np.array_equal(ro.counts()[0], r1.counts()[0])
    # two shards (env_offset = half the batch) sum to the unsharded counts
    shards = [_env(name, e // 2, 0.02, "A", st[k * e // 2:(k + 1) * e // 2], env_offset=k * e // 2) for k in range(2)]
    recs = [StateRecorder(s, genes=genes) for s in shards]
    for s, r in zip(shards, recs):
        s.rollout(3, recorder=r)
    torch.cuda.synchronize()
    for k in range(2):
        assert np.array_equal(recs[0].counts()[k] + recs[1].counts()[k], r1.counts()[k])
    for x in [whole, twin, only_hist, only_on] + shards:
        x.close()


def test_fused_recorder_equals_steady_state_histogram():
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200.discover import steady_state_histogram, steady_state_statistics
    name, e = "pbn28", 5000
    genes = [27, 3, 14, 0, 21]
    envs = [VecPBNEnv(product_net(name), e, None, device="cuda:0", perturb_p=0.01, seed=5, horizon=0) for _ in range(2)]
    st = _start(name, e)
    import torch
    for env in envs:
        env.set_state(torch.from_numpy(st.astype(np.int64)), packed=True)
    ref = steady_state_histogram(envs[0], 20, genes=genes, burn_in=10)
    rec = steady_state_statistics(envs[1], 20, burn_in=10, genes=genes)
    hist = rec.counts()[1]
    assert ref == {b: int(c) for b, c in enumerate(hist) if c}
    assert torch.equal(envs[0].state, envs[1].state)
    for env in envs:
        env.close()


def test_policy_loop_and_scalar_fallback():
    import torch
    from oracle.record_oracle import record_states
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200.discover import StateRecorder, steady_state_statistics
    from pbn_rl_b200.evaluate import hamming_policy
    name, e = "pbn7", 1500
    genes = [6, 0, 3]
    pol = hamming_policy(3)
    mk = lambda **kw: VecPBNEnv(product_net(name), e, attractor_set(name), device="cuda:0", perturb_p=0.02, seed=3,
                               horizon=20, auto_reset=True, **kw)
    envs = [mk(), mk()]
    for env in envs:
        env.reset()
    rec = steady_state_statistics(envs[0], 9, burn_in=4, genes=genes, stride=2, policy=pol)
    on = np.zeros(7, dtype=np.uint64)
    hist = np.zeros(8, dtype=np.uint64)
    for s in range(1, 14):
        envs[1].step(pol(envs[1].observe()), stats=False)
        if s > 4 and (s - 4) % 2 == 0:
            a, b = record_states(envs[1].state.cpu().numpy().astype(np.uint64), 7, genes)
            on += a
            hist += b
    assert np.array_equal(rec.counts()[0], on) and np.array_equal(rec.counts()[1], hist) and rec.n == 4 * e
    # scalar kernel: rollout(recorder=) falls back to the step loop + pbn_record_states
    st = _start("pbn10", 777)
    sc = [_env("pbn10", 777, 0.05, "A", st, kernel="scalar") for _ in range(2)]
    assert sc[0].kernel == "scalar"
    r = StateRecorder(sc[0], genes=list(range(10)))
    sc[0].rollout(6, recorder=r, stride=3)
    on = np.zeros(10, dtype=np.uint64)
    hist = np.zeros(1024, dtype=np.uint64)
    for s in range(1, 7):
        sc[1].step(None)
        if s % 3 == 0:
            a, b = record_states(sc[1].state.cpu().numpy().astype(np.uint64), 10, list(range(10)))
            on += a
            hist += b
    torch.cuda.synchronize()
    assert torch.equal(sc[0].state, sc[1].state)
    assert np.array_equal(r.counts()[0], on) and np.array_equal(r.counts()[1], hist)
    for x in envs + sc:
        x.close()


def test_record_argument_errors():
    import torch
    from pbn_rl_b200._cabi import PbnError, check
    from pbn_rl_b200.discover import StateRecorder
    env = _env("pbn28", 2048, 0.0, "A", _start("pbn28", 2048))
    lib, h = env.lib, env._h
    acc = torch.zeros((1 << 13,), dtype=torch.int64, device="cuda:0")
    st = env.state.data_ptr()

    def roll(n_steps=2, env_offset=0, n_envs=2048, stride=1, genes=(1, 2), n_proj=None):
        g = (C.c_int32 * max(len(genes), 1))(*genes)
        return lib.pbn_rollout_record(h, st, n_steps, 0, env_offset, n_envs, stride, g,
                                      len(genes) if n_proj is None else n_proj, acc.data_ptr(), acc.data_ptr(), None,
                                      env._stream())

    def rec(genes=(1, 2), n_envs=2048):
        g = (C.c_int32 * max(len(genes), 1))(*genes)
        return lib.pbn_record_states(h, st, n_envs, g, len(genes), acc.data_ptr(), acc.data_ptr(), env._stream())

    bad_genes = [tuple(range(13)), (3, 3), (-1,), (28,)]
    for genes in bad_genes:
        for call in (roll, rec):
            with pytest.raises(PbnError) as ex:
                check(call(genes=genes))
            assert ex.value.message
    for kw in (dict(stride=0), dict(stride=-2), dict(n_steps=-1), dict(n_steps=1 << 31), dict(env_offset=100),
               dict(env_offset=-1024), dict(n_envs=-1)):
        with pytest.raises(PbnError):
            check(roll(**kw))
    with pytest.raises(PbnError):
        check(rec(n_envs=-1))
    with pytest.raises(ValueError):
        StateRecorder(env, genes=list(range(13)))
    with pytest.raises(ValueError):
        StateRecorder(env, genes=[2, 2])
    with pytest.raises(ValueError):
        env.rollout(2, recorder=StateRecorder(env, genes=[1]), stride=0)
    assert int(acc.abs().sum().item()) == 0      # nothing was recorded by a rejected call
    sc = _env("pbn10", 1024, 0.0, "A", _start("pbn10", 1024), kernel="scalar")
    g = (C.c_int32 * 1)(1)
    with pytest.raises(PbnError):
        check(sc.lib.pbn_rollout_record(sc._h, sc.state.data_ptr(), 2, 0, 0, 1024, 1, g, 1, acc.data_ptr(), None, None,
                                        sc._stream()))
    env.close()
    sc.close()


def _exact_chain(p):
    """128 x 128 transition matrix of Bittner-7 with perturbation model A at rate p."""
    net = product_net("pbn7")
    n = net.n_genes
    T = np.zeros((1 << n, 1 << n))
    for x in range(1 << n):
        bits = [(x >> g) & 1 for g in range(n)]
        dist = np.ones(1)
        idx = np.zeros(1, dtype=np.int64)
        for i, (fs, ps) in enumerate(zip(net.functions, net.probabilities)):
            p1 = sum(pr for f, pr in zip(fs, ps) if f(bits))
            idx = np.concatenate([idx, idx | (1 << i)])
            dist = np.concatenate([dist * (1 - p1), dist * p1])
        np.add.at(T[x], idx, dist * (1 - p) ** n)
        for m in range(1, 1 << n):
            k = bin(m).count("1")
            T[x, x ^ m] += p ** k * (1 - p) ** (n - k)
    return T


def test_statistics_against_the_exact_chain():
    """Bittner-7, model A, p = 0.05: one recorded update of 2^20 envs after a burn-in long enough for |lambda_2|^b <
    1e-6 matches the stationary distribution of the exact chain (chi-square, the bound of the next-state test)."""
    import torch
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200.discover import steady_state_statistics
    p, e = 0.05, 1 << 20
    T = _exact_chain(p)
    assert np.allclose(T.sum(axis=1), 1.0)
    w, v = np.linalg.eig(T.T)
    order = np.argsort(-np.abs(w))
    pi = np.real(v[:, order[0]])
    pi /= pi.sum()
    lam2 = float(np.abs(w[order[1]]))
    burn = int(np.ceil(np.log(1e-6) / np.log(lam2)))
    env = VecPBNEnv(product_net("pbn7"), e, None, device="cuda:0", perturb_p=p, perturb_mode="A", seed=11, horizon=0)
    env.state.zero_()
    rec = steady_state_statistics(env, 1, burn_in=burn, genes=list(range(7)))
    counts = rec.counts()[1].astype(float)
    assert counts.sum() == e
    chi2 = sum((counts[t] - e * pi[t]) ** 2 / (e * pi[t]) for t in range(128) if pi[t] > 0)
    df = int((pi > 0).sum()) - 1
    assert chi2 < df + 6 * np.sqrt(2 * df) + 10, (chi2, df, burn, lam2)
    marg = rec.marginals()
    exact = np.array([sum(pi[t] for t in range(128) if (t >> g) & 1) for g in range(7)])
    assert np.all(np.abs(marg - exact) < 6 * np.sqrt(exact * (1 - exact) / e) + 1e-9)
    env.close()
