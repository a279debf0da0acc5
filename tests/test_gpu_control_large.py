"""GPU: exact control at 21 to 28 genes, where every operator is cut into launches of 2^22 states (pbn_b200.cu,
kDpSliceStates) and the expect kernel enumerates up to 23 free genes in per-warp digit tables.  The references scale
to 2^28 states (tests/control_oracle.py): formula inputs evaluated only where they are gathered, successor sets
enumerated in chunks, K_p as a tensor product, brute force and classification at sampled states.  The samples hold
the first and last state of every launch of every loop, one state per reachable free-gene count (runs across the
gene 21/22 boundary and wrapping from the last gene to gene 0) and random states; test_samples_cover_every_launch
asserts that."""
import numpy as np
import pytest

import control_oracle as CO
from helpers import attractor_set, make_network, product_net, run_state, window_network

pytestmark = pytest.mark.gpu

SLICE = 1 << 22         # kDpSliceStates: states (or state pairs) per launch of every DP loop
KP_TILE_BITS = 10       # kKpTileBits: genes folded by dp_kp_low_kernel; higher genes run dp_kp_bit_kernel
TOL = 1e-12 * 0.5       # 1e-12 max|u|: the formula inputs lie in [-0.5, 0.5)

EXPECT_CASES = [(22, 3, 22), (23, 3, 23), (25, 6, 25), (26, 3, 26), (28, 3, 28)]
PERT_CASES = [("window", 23), ("window", 24), ("make_network", 24)]
IMPROVE_N = [23, 24, 28]
SPREAD = (0, 1, 5, 13, 21, 22, 23, 25, 26, 27)   # 10 flip genes over both ends of the index
W_KINDS = {"ties": (CO.w_ties, -1.0), "rounding": (CO.w_rounding, -0.75), "normal": (CO.u_hash, -0.1)}


# ---- the samples ----------------------------------------------------------------------------------------------------
def slice_bounds(n):
    """First and last state of every launch of the expect, mix and improve loops."""
    S = 1 << n
    return {x for s0 in range(0, S, SLICE) for x in (s0, min(s0 + SLICE, S) - 1)}


def kp_bounds(n):
    """First and last state of every dp_kp_low_kernel launch, and the two states of the first and last pair of every
    dp_kp_bit_kernel slice of every gene it runs."""
    S = 1 << n
    out = set(slice_bounds(n))
    for b in range(min(n, KP_TILE_BITS), n):
        for j0 in range(0, S // 2, SLICE):
            for j in (j0, min(j0 + SLICE, S // 2) - 1):
                lo = ((j >> b) << (b + 1)) | (j & ((1 << b) - 1))
                out |= {lo, lo | (1 << b)}
    return out


def window_states(n, k, seed):
    """Slice bounds, the all-ones state (n free genes), one run per free count 0..n-k across genes 21/22 and one
    wrapping n-1 -> 0, and 64 random states."""
    st = slice_bounds(n) | {0, (1 << n) - 1}
    for f in range(0, n - k + 1):
        length = f + k - 1 if f else k - 1
        st.add(run_state(n, 22 - length // 2, length))
        st.add(run_state(n, n - length // 2, length))
    st |= set(np.random.default_rng(seed).choice(1 << n, size=64, replace=False).tolist())
    return np.array(sorted(st), dtype=np.int64)


def digits(free):
    """Digit tables of dp_expect_kernel in use for a state with ``free`` free genes (5 spread over the lanes)."""
    return (max(free - 5, 0) + 3) // 4


def improve_states(n, seed):
    st = slice_bounds(n) | {0, (1 << n) - 1, (1 << (n - 1)) - 1, 1 << (n - 1)}
    st |= set(np.random.default_rng(seed).choice(1 << n, size=64, replace=False).tolist())
    return np.array(sorted(st), dtype=np.int64)


# ---- networks and handles -------------------------------------------------------------------------------------------
def _window(n, k, seed):
    from pbn_rl_b200 import PBNNetwork
    return PBNNetwork.from_expressions(*window_network(n, k, seed))


def _make24():
    from pbn_rl_b200 import PBNNetwork
    return PBNNetwork.from_expressions(*make_network(24, 2, 3, seed=24))


def _env(net, mode="A", p=0.0, attractors=None, **kw):
    from pbn_rl_b200 import AttractorSet, VecPBNEnv
    n = net.n_genes
    if attractors is None:
        attractors = AttractorSet([[tuple([0] * n)]], n)
    kw.setdefault("kernel", "scalar")
    return VecPBNEnv(net, 1, attractors, device="cuda:0", perturb_mode=mode, perturb_p=p, **kw)


def _formula(f, n):
    import torch
    return f(torch.arange(1 << n, dtype=torch.int64, device="cuda:0"))


def _same_bits(a, b):
    import torch
    return torch.equal(a.view(torch.int64) if a.dtype == torch.float64 else a,
                       b.view(torch.int64) if b.dtype == torch.float64 else b)


def _release():
    import torch
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _gather(x, states):
    import torch
    return x[torch.from_numpy(states).to(x.device)].cpu().numpy()


# ---- 1. expect at p = 0 on window networks --------------------------------------------------------------------------
@pytest.mark.parametrize("n,k,seed", EXPECT_CASES)
def test_expect_window_network(n, k, seed):
    """(F u) at every launch's first and last state, every reachable free count (every digit count and partial last
    digit of the expect kernel) and random states, against the chunked successor enumeration; a second call is
    bit-identical."""
    from pbn_rl_b200.control import _Backup
    net = _window(n, k, seed)
    env = _env(net)
    bk = _Backup(env)
    states = window_states(n, k, seed)
    u = _formula(CO.u_hash, n)
    w = bk.expect(u)
    got = _gather(w, states)
    assert _same_bits(w, bk.expect(u))
    del u, w
    bk = None
    env.close()
    _release()
    want = CO.sparse_expect(net, CO.u_hash, states)
    err = np.abs(got - want)
    i = int(err.argmax())
    assert err[i] <= TOL, (int(states[i]), int(CO.free_counts(net, states[i:i + 1])[0]), got[i], want[i])


# ---- 2. expect with perturbation at 23 and 24 genes ------------------------------------------------------------------
@pytest.mark.parametrize("kind,n", PERT_CASES)
def test_expect_perturbed(kind, n):
    """Models A and B at p = 1e-3, 0.05, 0.3: every dp_kp_low_kernel launch, every dp_kp_bit_kernel slice of every
    higher gene and every mix launch, against K_p as a tensor product (itself checked against the per-mask sum)."""
    from pbn_rl_b200.control import _Backup
    net = _window(n, 3, n) if kind == "window" else _make24()
    states = np.array(sorted(set(window_states(n, 3, n).tolist()) | kp_bounds(n)), dtype=np.int64)
    s_all = np.arange(1 << n, dtype=np.int64)
    u_host = CO.u_hash(s_all)
    fu = CO.sparse_expect(net, u_host, states)
    for p in (1e-3, 0.05, 0.3):
        kpu = CO.kp_tensor(u_host, p)
        if p == 0.05:
            few = states[[0, len(states) // 2, -1]]
            assert np.abs(kpu[few] - CO.kp_direct(u_host, few, p)).max() <= 1e-14
        c = (1.0 - p) ** n
        want = {"A": c * fu + kpu[states] - c * u_host[states], "B": CO.sparse_expect(net, kpu, states)}
        for mode in ("A", "B"):
            env = _env(net, mode, p)
            bk = _Backup(env)
            u = _formula(CO.u_hash, n)
            w = bk.expect(u)
            got = _gather(w, states)
            assert _same_bits(w, bk.expect(u)), (mode, p)
            del u, w
            bk = None
            env.close()
            err = np.abs(got - want[mode])
            i = int(err.argmax())
            assert err[i] <= TOL, (mode, p, int(states[i]), got[i], want[mode][i])
    _release()


# ---- 3. Bittner-28 ---------------------------------------------------------------------------------------------------
def _bittner28_states(env, seed=28):
    """The state with the most free genes (found with pbn_successor_sets over all 2^28 states), the slice bounds and
    64 random states.  The successor sets only choose the states: the reference recomputes them."""
    import torch
    n, S = env.n_genes, 1 << env.n_genes
    c1 = torch.empty((SLICE, 1), dtype=torch.int64, device=env.device)
    c0 = torch.empty_like(c1)
    best, best_state = -1, -1
    for s0 in range(0, S, SLICE):
        st = torch.arange(s0, s0 + SLICE, dtype=torch.int64, device=env.device).unsqueeze(1)
        assert env.lib.pbn_successor_sets(env._h, st.data_ptr(), SLICE, c1.data_ptr(), c0.data_ptr(),
                                          env._stream()) == 0
        fr = c1[:, 0] & c0[:, 0]
        pc = torch.zeros(SLICE, dtype=torch.int64, device=env.device)
        for i in range(n):
            pc += (fr >> i) & 1
        j = int(pc.argmax().item())
        if int(pc[j].item()) > best:
            best, best_state = int(pc[j].item()), s0 + j
    st = slice_bounds(n) | {best_state}
    st |= set(np.random.default_rng(seed).choice(S, size=64, replace=False).tolist())
    return np.array(sorted(st), dtype=np.int64), best_state, best


def test_expect_bittner28():
    """Bittner-28 at p = 0, the network exact control is for: its state with the most free genes (23), every launch's
    first and last state and random states against the chunked successor enumeration; deterministic; the workspace
    at the largest admitted size."""
    from pbn_rl_b200.control import _Backup
    net = product_net("pbn28")
    env = _env(net, attractors=attractor_set("pbn28"))
    assert env.lib.pbn_dp_workspace_bytes(env._h) == 24 << 28
    states, top, top_free = _bittner28_states(env)
    assert top_free == 23 and int(CO.free_counts(net, [top])[0]) == 23
    bk = _Backup(env)
    u = _formula(CO.u_hash, 28)
    w = bk.expect(u)
    got = _gather(w, states)
    assert _same_bits(w, bk.expect(u))
    del u, w
    bk = None
    env.close()
    _release()
    want = CO.sparse_expect(net, CO.u_hash, states)
    err = np.abs(got - want)
    i = int(err.argmax())
    assert err[i] <= TOL, (int(states[i]), got[i], want[i])


# ---- 4. improve at 23, 24, 28 genes ----------------------------------------------------------------------------------
def _flip_sets(n):
    spread = sum(1 << g for g in SPREAD if g < n)
    return [((1 << n) - 1, k) for k in range(0, 4)] + [(spread, k) for k in range(0, 9)]


@pytest.mark.parametrize("kind", sorted(W_KINDS))
@pytest.mark.parametrize("n", IMPROVE_N)
def test_improve_large(n, kind):
    """Values and policies at sampled states bit-identical to brute force with the contract's tie order, for every
    gene with up to 3 flips and for 10 genes at both ends of the index with 0..8 flips, where the neighbours of a
    state through genes >= 22 lie in other launches; a second call is bit-identical."""
    from pbn_rl_b200.control import _Backup
    f, r_action = W_KINDS[kind]
    env = _env(_window(n, 3, n))
    bk = _Backup(env)
    w = _formula(f, n)
    states = improve_states(n, n)
    for genes, kmax in _flip_sets(n):
        v, pol = bk.improve(w, genes, kmax, r_action)
        gv, gp = _gather(v, states), _gather(pol, states).astype(np.int64)
        v2, p2 = bk.improve(w, genes, kmax, r_action)
        assert _same_bits(v, v2) and _same_bits(pol, p2), (genes, kmax)
        del v, pol, v2, p2
        bv, bp = CO.improve_brute_states(f, states, genes, kmax, r_action)
        assert np.array_equal(gv.view(np.uint64), bv.view(np.uint64)), (hex(genes), kmax)
        assert np.array_equal(gp, bp), (hex(genes), kmax)
    del w
    bk = None
    env.close()
    _release()


# ---- 5. the pipeline at 24 genes ------------------------------------------------------------------------------------
def _attractors24():
    """Single-state targets in different launches, and two targets of several entries with '*' genes (the
    multi-entry path of pbn_in_target / pbn_attractor_id), one spread over every launch through genes 22 and 23."""
    from pbn_rl_b200 import AttractorSet

    def bits(s):
        return tuple((s >> i) & 1 for i in range(24))

    def star(s, genes):
        return tuple("*" if i in genes else (s >> i) & 1 for i in range(24))

    return AttractorSet([[star(0x2C5A17, {0, 1, 2, 3, 22, 23}), star(0x913F0E, {5, 9, 23})],
                         [bits(0x5A5A5A)],
                         [bits(0x0F0F0F)],
                         [bits(0xC00001), star(0x8421F0, {4, 11, 17}), bits(0x7FFFFF)]], 24)


def _members(attrs, seed):
    """A few states of every entry (its '*' genes drawn at random) and the entry with every '*' at 0 and at 1."""
    rng = np.random.default_rng(seed)
    out = set()
    for attr in attrs.attractors:
        for e in attr:
            stars = [i for i, b in enumerate(e) if b == "*"]
            base = sum(1 << i for i, b in enumerate(e) if b == 1)
            out |= {base, base | sum(1 << i for i in stars)}
            for _ in range(4):
                out.add(base | sum(1 << i for i in stars if rng.integers(0, 2)))
    return out


def pipeline_states(attrs):
    st = slice_bounds(24) | _members(attrs, 24)
    st |= set(np.random.default_rng(240).choice(1 << 24, size=64, replace=False).tolist())
    return np.array(sorted(st), dtype=np.int64)


def test_classify_24():
    """_Backup.classify (pbn_in_target / pbn_attractor_id in launches of 2^22 states) equals the reference at the
    members of every attractor entry, every launch's first and last state and random states."""
    from pbn_rl_b200.control import _Backup
    attrs = _attractors24()
    env = _env(_make24(), attractors=attrs)
    bk = _Backup(env)
    states = pipeline_states(attrs)
    for t in range(len(attrs)):
        hit, wrong = bk.classify(t)
        h_ref, w_ref = CO.classify_states(24, attrs.attractors, t, states)
        assert np.array_equal(_gather(hit, states), h_ref), t
        assert np.array_equal(_gather(wrong, states), w_ref), t
        assert h_ref.any() and w_ref.any()
    bk = None
    env.close()
    _release()


# flips are cheap against the success reward, so the optimal policies flip genes in every launch
_RETURN_KW = dict(horizon=10, bins=3, r_success=10.0, r_step=-0.25, r_action=-0.1, r_wrong=-2.0)


def _near_target(attrs, seed):
    """Four start states two flips away from members of target 0's entries, in launches 1, 2 and 3."""
    rng = np.random.default_rng(seed)
    out = []
    for e, hi in ((0, 1), (0, 2), (0, 3), (1, 2)):
        entry = attrs.attractors[0][e]
        s = sum(1 << i for i, b in enumerate(entry) if b == 1)
        s |= sum(1 << i for i, b in enumerate(entry) if b == "*" and i < 22 and rng.integers(0, 2))
        if entry[22] == "*":
            s |= (hi & 1) << 22
        if entry[23] == "*":
            s |= (hi >> 1) << 23
        fixed = [i for i, b in enumerate(entry) if b != "*" and i < 22]
        for i in rng.choice(fixed, size=2, replace=False):
            s ^= 1 << int(i)
        out.append(s)
    return out


@pytest.mark.parametrize("objective", ["return", "steps"])
def test_policy_values_of_the_optimum_24(objective):
    """policy_values of the optimal per-stage policies equals solve_control's values bit for bit at every stage over
    all 2^24 states: both add r_step + (fl(r_action k) + w[s ^ m]) in the same order, so any state or slice slip in
    the policy improve writes shows up."""
    import torch
    from pbn_rl_b200 import policy_values, solve_control
    attrs = _attractors24()
    env = _env(_make24(), "A", 0.01, attractors=attrs, **_RETURN_KW)
    stages = 10 if objective == "return" else 4
    for target in (0, 3):
        sol = solve_control(env, target, objective=objective, stages=stages)
        assert sol.values.shape == (stages + 1, 1 << 24)
        assert bool((sol.policies != 0).any()) and bool((sol.policies[:, 1 << 23:] != 0).any())
        pv = policy_values(env, target, sol.policies, objective=objective, stages=stages)
        for k in range(stages + 1):
            assert torch.equal(pv[k].view(torch.int64), sol.values[k].view(torch.int64)), (target, k)
        del sol, pv
    env.close()
    _release()


@pytest.mark.parametrize("mode,p", [("A", 0.0), ("A", 0.01)])
def test_return_rollouts_24(mode, p):
    """VecPBNEnv rollouts of the optimal "return" policy (horizon 10) from start states two flips away from the
    target in launches 1..3: the mean return of 2^14 envs per start lies within 5 sigma of V_10."""
    import torch
    from pbn_rl_b200 import VecPBNEnv, solve_control
    net, attrs = _make24(), _attractors24()
    kw = dict(_RETURN_KW, perturb_p=p, perturb_mode=mode, kernel="scalar")
    solver = VecPBNEnv(net, 1, attrs, device="cuda:0", **kw)
    target = 0
    sol = solve_control(solver, target)
    starts = _near_target(attrs, 24)
    assert sorted({s // SLICE for s in starts}) == [1, 2, 3]
    assert not CO.classify_states(24, attrs.attractors, target, starts)[0].any()
    per = 1 << 14
    e = per * len(starts)
    env = VecPBNEnv(net, e, attrs, device="cuda:0", seed=77, **kw)
    env.set_state(torch.tensor(starts, dtype=torch.int64, device="cuda:0").repeat_interleave(per).unsqueeze(1),
                  packed=True)
    env.set_target(torch.full((e,), target, dtype=torch.int32))
    env.t.zero_()
    ret = torch.zeros(e, dtype=torch.float64, device="cuda:0")
    active = torch.ones(e, dtype=torch.bool, device="cuda:0")
    for t in range(10):
        env.step(sol.actions(env.state, steps_left=10 - t))
        ret += torch.where(active, env.reward.to(torch.float64), 0.0)
        active &= ~(env.terminated.bool() | env.truncated.bool())
    assert not bool(active.any())
    r = ret.cpu().numpy().reshape(len(starts), per)
    v = sol.value(torch.tensor(starts), steps_left=10).cpu().numpy()
    sem = r.std(axis=1, ddof=1) / np.sqrt(per)
    if p > 0.0:     # the returns vary, so the comparison is not decided by unobserved rare events
        assert np.all(sem > 1e-3), sem
    assert np.all(np.abs(r.mean(axis=1) - v) <= 5 * sem + 1e-9), (r.mean(axis=1), v, sem)
    env.close()
    solver.close()
    _release()


# ---- what the samples reach ------------------------------------------------------------------------------------------
def test_samples_cover_every_launch():
    """The samples above hold a state of 26 or more free genes, every digit count 0..6 of the expect kernel, and the
    first and last state of every launch of every DP loop at every size they run."""
    seen_digits, top = set(), 0
    for n, k, seed in EXPECT_CASES:
        states = window_states(n, k, seed)
        assert slice_bounds(n) <= set(states.tolist())
        fc = CO.free_counts(_window(n, k, seed), states)
        top = max(top, int(fc.max()))
        seen_digits |= {digits(int(f)) for f in fc}
        assert set(range(0, n - k + 1)) | {n} == set(fc.tolist())
    assert top >= 26 and seen_digits == set(range(7))
    for kind, n in PERT_CASES:
        states = set(window_states(n, 3, n).tolist()) | kp_bounds(n)
        assert kp_bounds(n) <= states and slice_bounds(n) <= states and (1 << n) // SLICE >= 2
    assert any((1 << (n - 1)) // SLICE >= 2 for _, n in PERT_CASES)     # dp_kp_bit_kernel runs more than one slice
    for n in IMPROVE_N:
        assert slice_bounds(n) <= set(improve_states(n, n).tolist()) and (1 << n) // SLICE >= 2
    attrs = _attractors24()
    states = pipeline_states(attrs)
    assert slice_bounds(24) <= set(states.tolist())
    assert {int(s) // SLICE for s in _members(attrs, 24)} == {0, 1, 2, 3}
