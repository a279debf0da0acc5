"""GPU: edge cases of the plane-resident step and the recording rollout, and contract edges of every kernel.

- The plane-resident step on every synthetic network it accepts (1..96 genes, 1..8 action bytes, wide and weighted
  predictors), against the oracle and against the row-format kernel with auto-reset; its refusals.
- Attractor-table limits of the plane-resident step: 254 attractors, 256 multi-state entries, target ids past the table.
- Action bytes above N (no-ops that do not count towards the reward) and the saturating episode counter on the
  scalar, row-format and plane-resident kernels.
- The recording rollout on every synthetic network the sliced kernel accepts, against oracle/record_oracle.py.
- Long single-tile rollouts: the perturbation count of one call past 2^32, the in-tile flush of the recorded counts.
- Rollout statistics over ragged batches.
Networks are the parametrization; the other axes loop inside a test, so each network's NVRTC programs are built once."""
import time

import numpy as np
import pytest

from helpers import CASES, attractor_set, make_attractors, make_network, oracle_net, product_net

pytestmark = pytest.mark.gpu

MODES = {"none": 0, "A": 1, "B": 2, "C": 3}
KW = dict(r_success=2.5, r_step=-0.5, r_action=-1.0)
SEED = 4242
SLICED = [c[:5] for c in CASES if "sliced" in c[5]]
RESIDENT = [c for c in SLICED if c[1] <= 4]      # more than 4 predictors per gene: row-format kernels only
REFUSED = [c for c in SLICED if c[1] > 4]


def _synthetic(n, kmax, amax, uniform):
    from oracle import pbn_oracle as O
    from pbn_rl_b200 import PBNNetwork
    genes, exprs = make_network(n, kmax, amax, seed=1000 + n, uniform=uniform)
    return PBNNetwork.from_expressions(genes, exprs), O.OracleNetwork(genes, exprs), exprs


def _states(rng, e, net):
    masks = np.array(net.state_mask(), dtype=np.uint64)
    w = net.n_words
    return ((rng.integers(0, 2**63, size=(e, w), dtype=np.int64).astype(np.uint64) * np.uint64(2))
            + rng.integers(0, 2, size=(e, w)).astype(np.uint64)) & masks


def _env(net, e, aset, mode="A", p=0.0, bins=3, kernel="sliced", resident=False, **kw):
    from pbn_rl_b200 import VecPBNEnv
    args = dict(KW)
    args.update(kw)
    env = VecPBNEnv(net, e, aset, device="cuda:0", perturb_p=p, perturb_mode=mode, seed=SEED, bins=bins,
                    kernel=kernel, resident=resident, **args)
    assert env.kernel == kernel
    return env


def _load(env, state, target=None, t=None):
    import torch
    env.set_state(torch.from_numpy(state.astype(np.int64)), packed=True)
    if target is not None:
        env.set_target(torch.from_numpy(np.asarray(target, dtype=np.int32)))
    if t is not None:
        env.t.copy_(torch.from_numpy(np.asarray(t, dtype=np.uint16).view(np.int16)))


def _compare(env, expect, tag):
    import torch
    torch.cuda.synchronize()
    nxt, t1, rew, term, trunc = expect
    assert np.array_equal(env.reward.cpu().numpy().view(np.uint32), rew.view(np.uint32)), tag + ": reward"
    assert np.array_equal(env.terminated.cpu().numpy(), term), tag + ": terminated"
    assert np.array_equal(env.truncated.cpu().numpy(), trunc), tag + ": truncated"
    assert np.array_equal(env.state.cpu().numpy().astype(np.uint64), nxt), tag + ": state"
    assert np.array_equal(env.t.cpu().numpy().astype(np.uint16), t1), tag + ": t"


def _no_target(x, n_attr):
    """Target ids as the plane-resident export writes them: negative or >= the table size -> -1."""
    x = np.asarray(x)
    return np.where((x >= 0) & (x < n_attr), x, -1)


def _twins(envs, acts, n_attr, tag):
    """Step a plane-resident env and its row-format twin with the same actions: every output of every step, then
    state, target, source, counters and statistics are identical."""
    import torch
    for step, a in enumerate(acts):
        outs = []
        for env in envs:
            env.step(a)
            outs.append((env.reward.view(torch.int32).clone(), env.terminated.clone(), env.truncated.clone(),
                         env.source_id.clone()))
        for k, (x, y) in enumerate(zip(*outs)):
            assert torch.equal(x, y), "%s: output %d differs at step %d" % (tag, k, step)
    torch.cuda.synchronize()
    assert torch.equal(envs[0].state, envs[1].state), tag + ": state"
    assert np.array_equal(envs[0].target_id.cpu().numpy(), _no_target(envs[1].target_id.cpu().numpy(), n_attr)), tag
    assert torch.equal(envs[0].t, envs[1].t), tag + ": t"
    s0, s1 = envs[0].stats(), envs[1].stats()
    assert s0 == s1, (tag, s0, s1)
    return s0


# ---------------------------------------------------------------------------------------------- plane-resident step
@pytest.mark.parametrize("n,kmax,amax,bins,uniform", RESIDENT)
def test_resident_synthetic_networks(n, kmax, amax, bins, uniform, monkeypatch):
    import torch
    from oracle import pbn_oracle as O
    from pbn_rl_b200 import AttractorSet
    net, onet, exprs = _synthetic(n, kmax, amax, uniform)
    attrs = make_attractors(n, 5, seed=n)
    aset = AttractorSet(attrs, n)
    tables = O.attractor_tables(attrs, n)
    pw = np.random.default_rng(n).random((5, 5))
    np.fill_diagonal(pw, 0.0)
    for e in (1500, 2048):
        rng = np.random.default_rng(n + e)
        w = net.n_words
        masks = np.array(net.state_mask(), dtype=np.uint64)
        state0 = _states(rng, e, net)
        target = rng.integers(-1, 5, size=e).astype(np.int32)
        acts = [rng.integers(0, n + 1, size=(e, bins), dtype=np.uint8) for _ in range(4)]
        sel_inj = np.stack([rng.integers(0, len(r), size=e) for r in exprs], axis=1).astype(np.uint8)
        pert_inj = ((rng.integers(0, 2**63, size=(e, w), dtype=np.int64).astype(np.uint64) & masks)
                    * (rng.random((e, 1)) < 0.3)).astype(np.uint64)
        ids = np.arange(e, dtype=np.uint64)
        for mode in MODES:
            p = 0.0 if mode == "none" else 0.03
            expect, state, t = [], state0, np.zeros(e, np.uint16)
            for step in range(4):
                sel, pert = (sel_inj, pert_inj) if step == 1 else O.sliced_stream(onet, p, ids, step, SEED)
                out = O.batched_step(onet, tables, state, acts[step], target, t, horizon=3, mode=MODES[mode], sel=sel,
                                     pert=pert, **KW)
                expect.append(out)
                state, t = out[0], out[1]
            for warps in ("4", "8"):
                monkeypatch.setenv("PBN_B200_PLANES_WARPS", warps)
                tag = "n=%d E=%d %s w%s" % (n, e, mode, warps)
                env = _env(net, e, aset, mode, p, bins, resident=True, horizon=3)
                _load(env, state0, target)
                for step in range(4):
                    if step == 1:
                        env.step_injected(torch.from_numpy(acts[1]), torch.from_numpy(sel_inj),
                                          torch.from_numpy(pert_inj.astype(np.int64)))
                    else:
                        env.step(torch.from_numpy(acts[step]).cuda())
                    _compare(env, expect[step], "%s step %d" % (tag, step))
                env.close()
                # auto-reset with pair weights: the resident block against the row-format kernel
                envs = [_env(net, e, aset, mode, p, bins, resident=r, horizon=3, auto_reset=True, pair_weights=pw)
                        for r in (True, False)]
                for x in envs:
                    _load(x, state0, target)
                g = np.random.default_rng(e)
                steps = [torch.from_numpy(g.integers(0, n + 1, size=(e, bins), dtype=np.uint8)).cuda() for _ in range(10)]
                s = _twins(envs, steps, 5, tag + " auto-reset")
                assert s["episodes"] > 0 and s["steps"] == 10 * e, (tag, s)
                for x in envs:
                    x.close()


@pytest.mark.parametrize("n,kmax,amax,bins,uniform", REFUSED)
def test_resident_refuses_more_than_4_predictors(n, kmax, amax, bins, uniform):
    import torch
    from pbn_rl_b200 import AttractorSet
    net, _, exprs = _synthetic(n, kmax, amax, uniform)
    assert max(len(r) for r in exprs) > 4
    env = _env(net, 1024, AttractorSet(make_attractors(n, 5, seed=n), n), "A", 0.03, bins, resident=True)
    with pytest.raises(RuntimeError, match="more than 4 predictors"):
        env.step(torch.zeros((1024, bins), dtype=torch.uint8, device="cuda:0"))
    env.close()


def test_resident_refuses_wrong_attractor_reward():
    import torch
    env = _env(product_net("pbn28"), 1024, attractor_set("pbn28"), "A", 0.03, resident=True, r_wrong=-2.0)
    with pytest.raises(RuntimeError, match="r_wrong"):
        env.step(torch.zeros((1024, 3), dtype=torch.uint8, device="cuda:0"))
    env.close()


def _limit_table(multi, extra):
    """pbn28 tables at the resident kernel's limits, with its 14 real (single-state) attractors spread over the
    table so that envs reach their targets.  multi=False: 254 + extra single-state attractors; multi=True: attractors
    of 4 states (2 wildcards each, the first state real where there is one) in 256 + extra (care, value) entries."""
    rng = np.random.default_rng(254 + extra + 10 * multi)
    real = [a[0] for a in attractor_set("pbn28").attractors]
    count = 64 if multi else 254 + extra
    slots = np.linspace(0, count - 1, len(real)).astype(int)
    out = []
    for a in range(count):
        states = []
        for k in range(4 if multi else 1):
            if k == 0 and a in slots:
                states.append(tuple(real[list(slots).index(a)]))
                continue
            s = [int(v) for v in rng.integers(0, 2, size=28)]
            if multi:
                for j in rng.choice(28, size=2, replace=False):
                    s[int(j)] = "*"
            states.append(tuple(s))
        out.append(states)
    if multi and extra:
        out[-1].append(tuple("*" if j < 3 else 0 for j in range(28)))
    assert sum(len(a) for a in out) == (256 + extra if multi else 254 + extra)
    return out


@pytest.mark.parametrize("multi", [False, True])
def test_resident_attractor_table_limits(multi):
    import torch
    from pbn_rl_b200 import AttractorSet
    net, e = product_net("pbn28"), 2048 + 300
    attrs = _limit_table(multi, 0)
    aset = AttractorSet(attrs, 28)
    n_attr = len(attrs)
    rng = np.random.default_rng(5)
    state0 = _states(rng, e, net)
    real = np.array([sum(int(b) << i for i, b in enumerate(a[0]) if b != "*") for a in attractor_set("pbn28").attractors],
                    dtype=np.uint64)
    slots = np.linspace(0, n_attr - 1, len(real)).astype(np.int32)
    target = rng.integers(0, n_attr, size=e).astype(np.int32)
    start_real = rng.random(e) < 0.5                  # half the envs start in a real attractor, their target
    r = rng.integers(0, len(real), size=int(start_real.sum()))
    state0[start_real, 0] = real[r]
    target[start_real] = slots[r]
    special = np.array([-5, -1, 0, n_attr - 1, 254, 255, 1000], dtype=np.int32)
    target[::3] = special[rng.integers(0, len(special), size=len(target[::3]))]
    g = torch.Generator(device="cuda").manual_seed(3)
    # bytes 0..255: most are no-ops, so envs stay in their attractors
    acts = [torch.randint(0, 256, (e, 3), generator=g, device="cuda", dtype=torch.uint8) for _ in range(10)]
    envs = [_env(net, e, aset, "A", 0.03, resident=r, horizon=3, auto_reset=True) for r in (True, False)]
    for x in envs:
        _load(x, state0, target)
    s = _twins(envs, acts, n_attr, "multi" if multi else "254 attractors")
    assert s["terminated"] > 0 and s["truncated"] > 0, s
    for x in envs:
        x.close()
    # one attractor / one entry more is refused
    big = _env(net, 1024, AttractorSet(_limit_table(multi, 1), 28), "A", 0.03, resident=True)
    with pytest.raises(RuntimeError, match="entries > 256" if multi else "attractors > 254"):
        big.step(torch.zeros((1024, 3), dtype=torch.uint8, device="cuda:0"))
    big.close()


# ---------------------------------------------------------------------------------------------- every kernel
def _kernels():
    return [("scalar", False), ("sliced", False), ("sliced", True)]


@pytest.mark.parametrize("bins", [1, 3, 8])
def test_action_bytes_above_n_are_noops(bins):
    """Action bytes 0..255 -- repeats, 0, N, N + 1, 255 -- on the three kernels, bit for bit against the oracle."""
    import torch
    from oracle import pbn_oracle as O
    name, e, p = "pbn28", 2048 + 100, 0.03
    net, onet, n = product_net(name), oracle_net(name), 28
    tables = O.attractor_tables(attractor_set(name).attractors, n)
    rng = np.random.default_rng(bins)
    state0 = _states(rng, e, net)
    target = rng.integers(0, len(tables[0]) - 1, size=e).astype(np.int32)
    acts = rng.integers(0, 256, size=(e, bins)).astype(np.uint8)
    acts[0::8] = acts[0::8, :1]                                    # one value repeated in every byte
    acts[1::8, -1] = 0
    acts[2::8, 0] = n
    acts[3::8, 0] = n + 1
    acts[4::8] = 255
    acts[5::8] = n
    acts[6::8] = rng.integers(0, n + 1, size=(len(acts[6::8]), bins))
    acts[7::8, 0] = rng.integers(0, n + 1, size=len(acts[7::8]))  # one gene in range among bytes above N
    sel = np.stack([rng.integers(0, len(fs), size=e) for fs in net.functions], axis=1).astype(np.uint8)
    pert = np.where(rng.random((e, 1)) < 0.2, rng.integers(0, 1 << 28, size=(e, 1)), 0).astype(np.uint64)
    ids = np.arange(e, dtype=np.uint64)
    kw = dict(KW, horizon=20)
    for kernel, resident in _kernels():
        tag = "%s%s bins=%d" % (kernel, " resident" if resident else "", bins)
        env = _env(net, e, attractor_set(name), "A", p, bins, kernel, resident, horizon=20)
        _load(env, state0, target)
        state, t = state0, np.zeros(e, np.uint16)
        for step in range(2):
            a = acts if step == 0 else acts[::-1].copy()
            if step == 0:
                env.step_injected(torch.from_numpy(a), torch.from_numpy(sel), torch.from_numpy(pert.astype(np.int64)))
                s, q = sel, pert
            else:
                env.step(torch.from_numpy(a).cuda())
                if kernel == "scalar":
                    s, q = O.scalar_stream_selection(onet, ids, step, SEED), O.scalar_stream_perturbation(n, p, ids, step, SEED)
                else:
                    s, q = O.sliced_stream(onet, p, ids, step, SEED)
            out = O.batched_step(onet, tables, state, a, target, t, mode=1, sel=s, pert=q, **kw)
            _compare(env, out, "%s step %d" % (tag, step))
            state, t = out[0], out[1]
        flips = sum(bin(O.flip_mask_from_actions(r, n)).count("1") for r in acts) + \
            sum(bin(O.flip_mask_from_actions(r, n)).count("1") for r in acts[::-1])
        assert env.stats()["flips"] == flips, tag
        env.close()


@pytest.mark.parametrize("name", ["pbn28", "pbn70"])
def test_episode_counter_saturates(name):
    """t' = min(t + 1, 65535) against horizons 0, 1, 65534, 65535, with t in {0, 65533, 65534, 65535}: counters,
    flags, rewards and the episode statistics of two steps on the three kernels, against the oracle."""
    import torch
    from oracle import pbn_oracle as O
    e = 2048 + 64
    net, onet = product_net(name), oracle_net(name)
    n = net.n_genes
    rng = np.random.default_rng(n)
    state0 = _states(rng, e, net)
    t0 = np.array([0, 65533, 65534, 65535], dtype=np.uint16)[np.arange(e) % 4]
    acts = rng.integers(0, n + 1, size=(2, e, 3)).astype(np.uint8)
    sel = [np.stack([rng.integers(0, len(fs), size=e) for fs in net.functions], axis=1).astype(np.uint8)
           for _ in range(2)]
    pert = [np.zeros((e, net.n_words), dtype=np.uint64) for _ in range(2)]
    # targets that are reached: the attractors are the first step's next states of envs 0..15 (no actions), and every
    # fifth env repeats the inputs of one of them (with its own counter)
    acts[0, :16] = 0
    copy = np.arange(e) % 5 == 0
    src = np.arange(e)[copy] % 16
    for x in [state0, acts[0], sel[0]]:
        x[copy] = x[src]
    target = rng.integers(0, 16, size=e).astype(np.int32)
    target[:16] = np.arange(16)
    target[copy] = src
    nxt = onet.transition_batch(state0, np.zeros_like(state0), sel[0], pert[0], 1)
    from pbn_rl_b200 import AttractorSet
    aset = AttractorSet([[tuple(int(v) for v in ((int(nxt[k, i >> 6]) >> (i & 63)) & 1 for i in range(n)))]
                         for k in range(16)], n)
    tables = O.attractor_tables(aset.attractors, n)
    for horizon in (0, 1, 65534, 65535):
        expect, state, t = [], state0, t0
        for step in range(2):
            out = O.batched_step(onet, tables, state, acts[step], target, t, horizon=horizon, mode=1, sel=sel[step],
                                 pert=pert[step], **KW)
            expect.append(out)
            state, t = out[0], out[1]
        done = [(x[3] | x[4]).astype(bool) for x in expect]
        ref = dict(steps=2 * e, terminated=sum(int(x[3].sum()) for x in expect),
                   truncated=sum(int(x[4].sum()) for x in expect), episodes=sum(int(d.sum()) for d in done),
                   ep_len_sum=sum(int(x[1][d].astype(np.int64).sum()) for x, d in zip(expect, done)))
        if horizon in (1, 65534, 65535):
            assert ref["truncated"] > 0
        assert ref["terminated"] > 0
        for kernel, resident in _kernels():
            tag = "%s %s%s horizon=%d" % (name, kernel, " resident" if resident else "", horizon)
            env = _env(net, e, aset, "A", 0.0, 3, kernel, resident, horizon=horizon)
            _load(env, state0, target, t0)
            for step in range(2):
                env.step_injected(torch.from_numpy(acts[step]), torch.from_numpy(sel[step]),
                                  torch.from_numpy(pert[step].astype(np.int64)))
                _compare(env, expect[step], "%s step %d" % (tag, step))
            s = env.stats()
            assert {k: s[k] for k in ref} == ref, (tag, s, ref)
            env.close()


# ---------------------------------------------------------------------------------------------- recording rollout
def _projections(n, rng):
    edges = [g for g in (31, 32, 63, 64, 95) if g < n]
    genes = list(dict.fromkeys(edges + [n - 1, 0]))
    rest = [g for g in rng.permutation(n).tolist() if g not in genes]
    genes = (genes + rest)[:min(12, n)]
    rng.shuffle(genes)
    out = [[], [n - 1]]
    if n >= 12:
        out.append(genes)
    elif n > 1:
        out.append(genes)      # every gene: the largest projection a small network admits
    return out


@pytest.mark.parametrize("n,kmax,amax,bins,uniform", SLICED)
def test_rollout_record_synthetic_networks(n, kmax, amax, bins, uniform):
    from oracle import pbn_oracle as O
    from oracle.record_oracle import record_states
    from pbn_rl_b200.discover import StateRecorder
    net, onet, _ = _synthetic(n, kmax, amax, uniform)
    e, p, n_steps = 1500, 0.03, 7
    rng = np.random.default_rng(n)
    state = state0 = _states(rng, e, net)
    ids = np.arange(e, dtype=np.uint64)
    zero = np.zeros_like(state0)
    traj = []
    for step in range(n_steps):
        sel, pert = O.sliced_stream(onet, p, ids, step, SEED)
        state = onet.transition_batch(state, zero, sel, pert, O.PERT_A)
        traj.append(state.copy())
    for genes in _projections(n, rng):
        for stride in (1, 3, n_steps, n_steps + 1):
            recorded = [traj[s - 1] for s in range(1, n_steps + 1) if s % stride == 0]
            ref_on, ref_hist = np.zeros(n, dtype=np.uint64), np.zeros(1 << len(genes), dtype=np.uint64)
            for st in recorded:
                a, b = record_states(st, n, genes)
                ref_on += a
                ref_hist += b
            env = _env(net, e, None, "A", p, bins, horizon=0)
            _load(env, state0)
            rec = StateRecorder(env, genes=genes)
            env.rollout(n_steps, recorder=rec, stride=stride)
            on, hist = rec.counts()
            tag = (n, genes, stride)
            assert np.array_equal(env.state.cpu().numpy().astype(np.uint64), traj[-1]), tag
            assert np.array_equal(on, ref_on), tag
            assert np.array_equal(hist, ref_hist), tag
            assert rec.n == e * len(recorded)
            env.close()


# ---------------------------------------------------------------------------------------------- long single-tile runs
def test_rollout_perturbation_count_past_2_32():
    """One rollout of one 1024-env tile whose perturbation count exceeds 1.1 * 2^32 equals the same updates in calls of
    20000, and lies within 6 sigma of its expectation 1024 * N * p * n_steps."""
    import torch
    name, e, p, n_steps = "pbn70", 1024, 0.4, 170000
    net = product_net(name)
    start = _states(np.random.default_rng(1), e, net)
    envs = [_env(net, e, None, "A", p, horizon=0) for _ in range(2)]
    for x in envs:
        _load(x, start)
    t0 = time.time()
    envs[0].rollout(n_steps)
    torch.cuda.synchronize()
    t1 = time.time()
    left = n_steps
    while left:
        envs[1].rollout(min(left, 20000))
        left -= min(left, 20000)
    torch.cuda.synchronize()
    print("one call %.1f s, split %.1f s" % (t1 - t0, time.time() - t1))
    s0, s1 = envs[0].stats(), envs[1].stats()
    mean = e * net.n_genes * p * n_steps
    assert mean >= 1.1 * 2**32
    print("perturbed: one call %d, split %d, expected %.0f" % (s0["perturbed"], s1["perturbed"], mean))
    assert torch.equal(envs[0].state, envs[1].state)
    assert s0 == s1, (s0, s1)
    assert s0["steps"] == e * n_steps
    assert abs(s0["perturbed"] - mean) < 6 * np.sqrt(mean * (1 - p)), (s0["perturbed"], mean)
    for x in envs:
        x.close()


def test_rollout_record_flush_past_2_32():
    """Identity network (every gene keeps its value), p = 0: 2^22 + 1000 recorded updates of one tile in one call cross
    the in-tile flush twice; every count is known exactly and exceeds 2^32."""
    import torch
    from pbn_rl_b200 import PBNNetwork
    from pbn_rl_b200.discover import StateRecorder
    n, e, n_steps = 8, 1024, (1 << 22) + 1000
    genes = ["x%d" % i for i in range(n)]
    net = PBNNetwork.from_expressions(genes, [[("( x%d )" % i, 1.0)] for i in range(n)])
    rng = np.random.default_rng(8)
    state = rng.integers(0, 1 << n, size=(e, 1)).astype(np.uint64) | np.uint64(0x81)   # genes 0 and 7 on everywhere
    bits = (state[:, 0:1] >> np.arange(n, dtype=np.uint64)) & np.uint64(1)
    for proj in ([], [7, 0]):
        env = _env(net, e, None, "A", 0.0, horizon=0)
        _load(env, state)
        rec = StateRecorder(env, genes=proj)
        t0 = time.time()
        env.rollout(n_steps, recorder=rec, stride=1)
        torch.cuda.synchronize()
        print("proj %s: %.1f s" % (proj, time.time() - t0))
        on, hist = rec.counts()
        assert np.array_equal(env.state.cpu().numpy().astype(np.uint64), state)
        assert np.array_equal(on, bits.sum(axis=0).astype(np.uint64) * np.uint64(n_steps)), proj
        idx = np.zeros(e, dtype=np.int64)
        for j, g in enumerate(proj):
            idx |= bits[:, g].astype(np.int64) << j
        ref = np.bincount(idx, minlength=1 << len(proj)).astype(np.uint64) * np.uint64(n_steps)
        assert np.array_equal(hist, ref), proj
        assert int(on[0]) == e * n_steps > 2**32 and int(hist.max()) > 2**32
        env.close()


# ---------------------------------------------------------------------------------------------- ragged statistics
@pytest.mark.parametrize("e", [33, 4096 + 37])
def test_rollout_statistics_ragged_batches(e):
    import torch
    net = product_net("pbn28")
    start = _states(np.random.default_rng(e), e, net)
    for mode, p in (("A", 0.03), ("B", 0.03), ("C", 0.03), ("A", 0.4)):
        ref, dut = (_env(net, e, None, mode, p, horizon=0) for _ in range(2))
        for x in (ref, dut):
            _load(x, start)
        for _ in range(12):
            ref.step(None)
        dut.rollout(5)
        dut.rollout(7)
        torch.cuda.synchronize()
        assert torch.equal(ref.state, dut.state), (e, mode, p)
        s0, s1 = ref.stats(), dut.stats()
        assert s1["steps"] == s0["steps"] == 12 * e and s1["perturbed"] == s0["perturbed"] > 0, (e, mode, p, s0, s1)
        for x in (ref, dut):
            x.close()
