"""GPU: exhaustive attractor search (pbn_reach_mark / pbn_reach_sweep, discover.find_attractors_exhaustive).

The sweep's fixed point is checked bit for bit against the numpy restatement (tests/reach_oracle.py); the search
against the exhaustive host Tarjan (find_attractors_stg) up to 16 genes, and at 20 to 28 genes (Bittner-28 included)
against the rollout search and closure / strong-connectivity checks under the oracle's transition relation."""
import numpy as np
import pytest

import reach_oracle as RO
from helpers import golden, make_network, oracle_net, product_net

pytestmark = pytest.mark.gpu

MADE = {  # name -> make_network(n, kmax, amax, seed)
    "n3": (3, 2, 2, 3), "n5": (5, 2, 2, 5), "n6": (6, 2, 2, 7), "n9": (9, 2, 3, 9), "n12": (12, 3, 2, 13),
    "wide12": (12, 3, 12, 7), "n16": (16, 2, 4, 1), "n20": (20, 2, 3, 21), "n24": (24, 2, 3, 25),
    "dense20": (20, 3, 4, 20),
}


def trap_network(n):
    """Genes 0..n-3 keep x_i & x_(i+-1) (a zero spreads, so 'all ones' is reached only from itself); genes n-2, n-1
    swap.  Attractors: (all zeros | all ones) x (00, 11, the 01 <-> 10 cycle): three of the six have basins of one or
    two states, which uniform rollouts almost never hit."""
    k = n - 2
    genes = ["x%d" % i for i in range(n)]
    exprs = [[("( x%d & x%d )" % (i, (i + 1) % k), 0.5), ("( x%d & x%d )" % (i, (i - 1) % k), 0.5)] for i in range(k)]
    exprs += [[("x%d" % (n - 1), 1.0)], [("x%d" % (n - 2), 1.0)]]
    return genes, exprs


def _spec(name):
    if name.startswith("trap"):
        return trap_network(int(name[4:]))
    spec = MADE[name]
    return make_network(spec[0], spec[1], spec[2], seed=spec[3])


def _net(name):
    from pbn_rl_b200 import PBNNetwork
    if name in ("pbn7", "pbn10", "pbn28", "pbn70"):
        return product_net(name)
    return PBNNetwork.from_expressions(*_spec(name))


def _onet(name):
    from oracle.pbn_oracle import OracleNetwork
    if name in ("pbn7", "pbn10", "pbn28", "pbn70"):
        return oracle_net(name)
    return OracleNetwork(*_spec(name))


def _env(net, **kw):
    from pbn_rl_b200 import VecPBNEnv
    kw.setdefault("perturb_p", 0.0)
    return VecPBNEnv(net, 1024, None, device="cuda:0", horizon=0, bins=1, **kw)


def _marks(reach):
    return reach.marks.cpu().numpy().view(np.uint32).copy()


# ---- 1. the sweep against the oracle ----------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["pbn7", "pbn10", "n3", "n5", "n6", "n9", "n12", "wide12"])
def test_sweep_fixed_point_equals_oracle(name):
    from pbn_rl_b200 import find_attractors_stg
    from pbn_rl_b200.discover import ReachMarks
    net = _net(name)
    if name == "wide12":
        assert net.max_arity >= 7
    n, S = net.n_genes, 1 << net.n_genes
    succ = RO.successor_lists(net)
    sinks = find_attractors_stg(net)[1]["sink_sccs"]
    rng = np.random.default_rng(n)
    seed_sets = [[s for m in sinks for s in m], sinks[0], [int(x) for x in rng.integers(0, S, size=3)],
                 [int(x) for x in rng.integers(0, S, size=max(1, S // 16))], [S - 1]]
    env = _env(net)
    for seeds in seed_sets:
        reach = ReachMarks(env)
        first = reach.mark(list(seeds) + [S, S + 5, (1 << 40) + 1])       # states >= 2^N are ignored
        assert first == len(set(seeds))
        assert reach.mark(seeds) == 0                                    # already set: nothing counted
        reach.close()
        want = RO.backward_reach(succ, seeds)
        got = _marks(reach)
        assert np.array_equal(got, RO.pack_marks(want)), (name, seeds[:4])
        assert reach.count == int(want.sum()) == sum(bin(int(w)).count("1") for w in got)
        assert reach.sweep() == 0
    env.close()


def test_sweep_ignores_perturbation_probability():
    from pbn_rl_b200.discover import ReachMarks
    net = _net("pbn10")
    out = []
    for p in (0.0, 0.2):
        env = _env(net, perturb_p=p)
        reach = ReachMarks(env)
        reach.mark([0, 17])
        reach.close()
        out.append(_marks(reach))
        env.close()
    assert np.array_equal(out[0], out[1])
    assert np.array_equal(out[0], RO.pack_marks(RO.backward_reach(RO.successor_lists(net), [0, 17])))


# ---- 2./3. the search against the exhaustive host Tarjan -----------------------------------------------------------

@pytest.mark.parametrize("seed_rollouts", [0, 1 << 16])
@pytest.mark.parametrize("name", ["pbn7", "pbn10", "n12", "n16", "trap12", "trap16"])
def test_exhaustive_equals_tarjan(name, seed_rollouts):
    from pbn_rl_b200 import find_attractors_stg
    from pbn_rl_b200.discover import find_attractors_exhaustive
    net = _net(name)
    want, winfo = find_attractors_stg(net)
    got, info = find_attractors_exhaustive(net, seed_rollouts=seed_rollouts)
    assert info["states"] == winfo["sink_sccs"]
    assert got.attractors == want.attractors
    assert info["complete"] and info["uncovered"] == 0 and info["sweeps"] >= 1
    if seed_rollouts == 0:
        assert info["seeded"] == 0 and info["rounds"] >= 1
    if name in ("pbn7", "pbn10"):
        assert info["states"] == [sorted(m) for m in sorted(golden("k5_stg.json")[name]["sink_sccs"], key=min)]


def test_weak_seeding_misses_attractors_the_sweep_finds():
    """Three of trap16's six attractors have basins of one or two of the 65536 states: 1024 rollouts miss them, and
    the certificate finds them."""
    from pbn_rl_b200 import find_attractors_stg
    from pbn_rl_b200.discover import find_attractors_exhaustive, find_attractors_rollout
    net = _net("trap16")
    _, winfo = find_attractors_stg(net)
    assert len(winfo["sink_sccs"]) == 6
    _, rinfo = find_attractors_rollout(net, n_rollouts=1024)
    assert len(rinfo["states"]) < 6                                      # the seeding alone is incomplete
    got, info = find_attractors_exhaustive(net, seed_rollouts=1024)
    assert info["seeded"] == len(rinfo["states"]) and info["rounds"] >= 1
    assert info["states"] == winfo["sink_sccs"] and info["complete"]


# ---- 4. 20, 24 and 28 genes ----------------------------------------------------------------------------------------

def _descriptor(onet, s):
    """(can1, can0) of state s from the oracle: OR over 'every gene uses its predictor min(k, K_i - 1)'."""
    can1 = can0 = 0
    full = (1 << onet.n) - 1
    nf = [len(row) for row in onet.py_code]
    for k in range(max(nf)):
        t = onet.transition(s, 0, [min(k, nf[i] - 1) for i in range(onet.n)], 0)
        can1 |= t
        can0 |= ~t & full
    return can1, can0


def _assert_exact(onet, members_list):
    for members in members_list:
        mset = set(members)
        succ = {}
        for s in members[:64]:
            c1, c0 = _descriptor(onet, s)
            free = c1 & c0
            succ[s] = RO.enumerate_successors(c1 & ~free, free)
            assert set(succ[s]) <= mset, "attractor is not closed under the oracle's transition relation"
        if len(members) <= 64:           # strongly connected: everything is reached from the first member
            seen, todo = {members[0]}, [members[0]]
            while todo:
                for t in succ[todo.pop()]:
                    if t not in seen:
                        seen.add(t)
                        todo.append(t)
            assert seen == mset


@pytest.mark.parametrize("name", ["n20", "n24", "pbn28"])
def test_large_networks_complete(name):
    from pbn_rl_b200.discover import find_attractors_exhaustive, find_attractors_rollout
    net = _net(name)
    got, info = find_attractors_exhaustive(net)
    assert info["complete"] and info["uncovered"] == 0
    _, rinfo = find_attractors_rollout(net)
    assert {tuple(m) for m in rinfo["states"]} <= {tuple(m) for m in info["states"]}
    assert info["seeded"] == len(rinfo["states"])
    assert len(got) == len(info["states"]) >= 1
    assert [m[0] for m in info["states"]] == sorted(m[0] for m in info["states"])
    assert all(m == sorted(m) for m in info["states"])
    _assert_exact(_onet(name), info["states"])


# ---- 5. the incomplete path ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("seed_rollouts", [0, 4096])
def test_too_small_closure_limit_is_reported_incomplete(seed_rollouts):
    """pbn10's 11-state sink SCC does not fit a closure of 8 states: the search says so, the uncovered states are
    exactly those that reach none of the other attractors, and what it returns is exact."""
    from pbn_rl_b200.discover import find_attractors_exhaustive
    net = _net("pbn10")
    sinks = [sorted(m) for m in golden("k5_stg.json")["pbn10"]["sink_sccs"]]
    big = [m for m in sinks if len(m) == 11]
    assert len(big) == 1
    _, info = find_attractors_exhaustive(net, seed_rollouts=seed_rollouts, max_attractor_states=8)
    assert not info["complete"] and info["uncovered"] > 0
    assert info["states"] == sorted((m for m in sinks if len(m) != 11), key=lambda m: m[0])
    others = [s for m in info["states"] for s in m]
    assert info["uncovered"] == int((~RO.backward_reach(RO.successor_lists(net), others)).sum())


def test_attractor_larger_than_the_closure_limit_at_20_genes():
    """make_network(20, 3, 4, seed=20) has 5 to 16 free genes in every state; its attractor does not fit the default
    closure of 2^14 states, so the search ends incomplete (quickly: a round gives up after max_unresolved failed
    closures) and says so."""
    from pbn_rl_b200.discover import find_attractors_exhaustive
    net = _net("dense20")
    _, info = find_attractors_exhaustive(net)
    assert not info["complete"] and info["uncovered"] > 0 and info["rounds"] >= 1
    _assert_exact(_onet("dense20"), info["states"])


# ---- 6. determinism ------------------------------------------------------------------------------------------------

def test_marks_are_bit_identical_between_runs_at_24_genes():
    from pbn_rl_b200.discover import ReachMarks, find_attractors_exhaustive
    net = _net("n24")
    rng = np.random.default_rng(24)
    seeds = [int(x) for x in rng.integers(0, 1 << 24, size=5)]
    runs = []
    for _ in range(2):
        env = _env(net)
        reach = ReachMarks(env)
        reach.mark(seeds)
        reach.close()
        runs.append((_marks(reach), reach.count))
        env.close()
    assert np.array_equal(runs[0][0], runs[1][0]) and runs[0][1] == runs[1][1]
    assert runs[0][1] == sum(bin(int(w)).count("1") for w in runs[0][0])
    a = find_attractors_exhaustive(net)[1]
    b = find_attractors_exhaustive(net)[1]
    a.pop("sweeps"), b.pop("sweeps")     # how many sweeps a fixed point takes depends on timing, the fixed point does not
    assert a == b


# ---- 7. refusals ---------------------------------------------------------------------------------------------------

def test_refusals():
    import torch
    from pbn_rl_b200._cabi import PBN_ERR_INVALID, PBN_ERR_UNSUPPORTED, PbnError
    from pbn_rl_b200.discover import ReachMarks, find_attractors_exhaustive
    big = _env(_net("pbn70"))
    marks = torch.zeros((1 << 10,), dtype=torch.int32, device="cuda:0")
    newly = torch.zeros((1,), dtype=torch.int64, device="cuda:0")
    st = torch.zeros((4,), dtype=torch.int64, device="cuda:0")
    s = big._stream()
    assert big.lib.pbn_reach_sweep(big._h, marks.data_ptr(), newly.data_ptr(), s) == PBN_ERR_UNSUPPORTED
    assert big.lib.pbn_reach_mark(big._h, marks.data_ptr(), st.data_ptr(), 4, newly.data_ptr(), s) == PBN_ERR_UNSUPPORTED
    with pytest.raises(PbnError) as e:
        ReachMarks(big)
    assert e.value.code == PBN_ERR_UNSUPPORTED
    with pytest.raises(PbnError) as e:
        find_attractors_exhaustive(_net("pbn70"))
    assert e.value.code == PBN_ERR_UNSUPPORTED
    big.close()
    env = _env(_net("pbn10"))
    h, s, lib = env._h, env._stream(), env.lib
    assert lib.pbn_reach_sweep(h, None, newly.data_ptr(), s) == PBN_ERR_INVALID
    assert lib.pbn_reach_sweep(h, marks.data_ptr(), None, s) == PBN_ERR_INVALID
    assert lib.pbn_reach_sweep(None, marks.data_ptr(), newly.data_ptr(), s) == PBN_ERR_INVALID
    assert lib.pbn_reach_mark(h, None, st.data_ptr(), 4, newly.data_ptr(), s) == PBN_ERR_INVALID
    assert lib.pbn_reach_mark(h, marks.data_ptr(), st.data_ptr(), 4, None, s) == PBN_ERR_INVALID
    assert lib.pbn_reach_mark(h, marks.data_ptr(), None, 4, newly.data_ptr(), s) == PBN_ERR_INVALID
    assert lib.pbn_reach_mark(h, marks.data_ptr(), st.data_ptr(), -1, newly.data_ptr(), s) == PBN_ERR_INVALID
    assert lib.pbn_reach_mark(h, marks.data_ptr(), None, 0, newly.data_ptr(), s) == 0
    torch.cuda.synchronize()
    assert int(newly.item()) == 0 and int(marks.abs().sum().item()) == 0
    env.close()
