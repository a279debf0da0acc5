"""Exhaustive attractor search above 28 genes (pbn_reach_sweep with u64 state indices, N <= PBN_REACH_MAX_GENES = 34).

The sweep's marks are checked bit for bit over all 2^N states against analytic predicates: of trap networks at 29, 32,
33 and 34 genes (genes 32 and 33 evaluated by the second ballot), and of copy networks at 33 and 34 genes, whose fixed
point depends on free genes at 32 and above taking the value 1 as well as 0.  The search runs on trap33 / trap34 and on
bb33 (33 genes, a deterministic network) against the rollout search and the oracle's transition; the fixed point of a
deterministic random 33-gene network is checked against the oracle at sampled states.  CPU tests check both predicates
against the host fixed point (tests/reach_oracle.py)."""
import numpy as np
import pytest

import reach_oracle as RO
from helpers import GOLD, make_network

ATTRACTORS = [(ring, pair) for ring in ("zeros", "ones") for pair in ("00", "11", "cycle")]
PAIR_STATES = {"00": [0], "11": [3], "cycle": [1, 2]}


def trap_network(n):
    """Genes 0..n-3 keep x_i & x_(i+-1) (a zero spreads, so 'all ones' is reached only from itself); genes n-2, n-1
    swap.  Attractors: (all zeros | all ones) x (00, 11, the 01 <-> 10 cycle): three of the six have basins of one or
    two states, which uniform rollouts almost never hit."""
    k = n - 2
    genes = ["x%d" % i for i in range(n)]
    exprs = [[("( x%d & x%d )" % (i, (i + 1) % k), 0.5), ("( x%d & x%d )" % (i, (i - 1) % k), 0.5)] for i in range(k)]
    exprs += [[("x%d" % (n - 1), 1.0)], [("x%d" % (n - 2), 1.0)]]
    return genes, exprs


def pair_low_trap_network(n):
    """trap_network(n) with its genes permuted: the swap pair at genes 0, 1 and the ring at genes 2..n-1, so that free
    ring genes sit at gene 32 and above once n > 32."""
    genes, exprs = trap_network(n)
    order = [n - 2, n - 1] + list(range(n - 2))
    return [genes[i] for i in order], [exprs[i] for i in order]


def _layout(n, pair_low):
    """(first ring gene, first pair gene)."""
    return (2, 0) if pair_low else (0, n - 2)


def trap_attractor_states(n, pair_low, attractor):
    r0, p0 = _layout(n, pair_low)
    ring = 0 if attractor[0] == "zeros" else (1 << (n - 2)) - 1
    return [(ring << r0) | (p << p0) for p in PAIR_STATES[attractor[1]]]


def trap_reaches(states, n, pair_low, seeded):
    """bool tensor: which of ``states`` (an int64 tensor) reach one of the ``seeded`` attractors.  The ring and the pair
    evolve independently.  A ring part other than all ones reaches all zeros and never all ones; all ones reaches only
    itself.  The pair is deterministic and already in its attractor (00, 11 or the cycle).  So every state reaches
    exactly one attractor, (ring class, pair class), and that is a function of the state index."""
    r0, p0 = _layout(n, pair_low)
    full = (1 << (n - 2)) - 1
    ones = ((states >> r0) & full) == full
    pair = (states >> p0) & 3
    out = states < 0                        # all False, on the states' device
    for ring, pc in seeded:
        in_pair = (pair == 1) | (pair == 2) if pc == "cycle" else pair == PAIR_STATES[pc][0]
        out |= (ones if ring == "ones" else ~ones) & in_pair
    return out


def copy_network(n, u=6):
    """Genes 0..n-u-1 (n >= 2u) keep their value; gene n-u+j keeps its value or copies gene j (two predictors), so it
    is free exactly when it differs from gene j.  From s, a step (and so any number of steps) reaches every state with
    the low genes of s and, for each upper gene, its own value or its source's."""
    genes = ["x%d" % i for i in range(n)]
    exprs = [[("x%d" % i, 1.0)] for i in range(n - u)]
    exprs += [[("x%d" % (n - u + j), 0.5), ("x%d" % j, 0.5)] for j in range(u)]
    return genes, exprs


def copy_reaches(states, n, seeds, u=6):
    """bool tensor: which of ``states`` reach one of ``seeds`` in copy_network(n, u): the same low genes as a seed z, and
    every upper gene g equal to z's, unless z already has g equal to its source (then either value of g reaches z)."""
    low = (1 << (n - u)) - 1
    out = states < 0
    for z in seeds:
        m = (states & low) == (z & low)
        for j in range(u):
            g = n - u + j
            if (z >> g) & 1 != (z >> j) & 1:
                m &= ((states >> g) & 1) == (z >> g) & 1
        out |= m
    return out


def _net(genes_exprs):
    from pbn_rl_b200 import PBNNetwork
    return PBNNetwork.from_expressions(*genes_exprs)


def _trap(n, pair_low):
    return _net(pair_low_trap_network(n) if pair_low else trap_network(n))


def _env(net):
    from pbn_rl_b200 import VecPBNEnv
    return VecPBNEnv(net, 1024, None, device="cuda:0", horizon=0, bins=1, perturb_p=0.0)


# ---- CPU: the predicate against the host fixed point ---------------------------------------------------------------

@pytest.mark.parametrize("pair_low", [False, True])
@pytest.mark.parametrize("n", range(6, 13))
def test_trap_predicate_equals_backward_reach(n, pair_low):
    import torch
    succ = RO.successor_lists(_trap(n, pair_low))
    states = torch.arange(1 << n, dtype=torch.int64)
    subsets = [[a for a in ATTRACTORS if a != left] for left in ATTRACTORS] + [[a] for a in ATTRACTORS] + [ATTRACTORS]
    for seeded in subsets:
        seeds = [s for a in seeded for s in trap_attractor_states(n, pair_low, a)]
        want = RO.backward_reach(succ, seeds)
        assert np.array_equal(trap_reaches(states, n, pair_low, seeded).numpy(), want), (n, pair_low, seeded)


@pytest.mark.parametrize("n,u", [(8, 4), (10, 5), (12, 6)])
def test_copy_predicate_equals_backward_reach(n, u):
    import torch
    succ = RO.successor_lists(_net(copy_network(n, u)))
    states = torch.arange(1 << n, dtype=torch.int64)
    rng = np.random.default_rng(n)
    for seeds in ([0], [(1 << n) - 1], [int(x) for x in rng.integers(0, 1 << n, size=8)]):
        assert np.array_equal(copy_reaches(states, n, seeds, u).numpy(), RO.backward_reach(succ, seeds)), (n, seeds)


# ---- 1. analytic marks, bit for bit ----------------------------------------------------------------------------------

def _assert_marks(reach, n, predicate):
    """The device marks equal predicate(states) over all 2^N states, compared on the device in chunks of 2^26 states."""
    import torch
    dev = reach.marks.device
    weights = torch.ones(32, dtype=torch.int64, device=dev) << torch.arange(32, device=dev)
    chunk = min(1 << 26, 1 << n)
    total = 0
    for s0 in range(0, 1 << n, chunk):
        want = predicate(torch.arange(s0, s0 + chunk, dtype=torch.int64, device=dev))
        total += int(want.sum().item())
        want_words = (want.view(-1, 32).to(torch.int64) * weights).sum(1)
        got_words = reach.marks[s0 >> 5:(s0 + chunk) >> 5].to(torch.int64) & 0xFFFFFFFF
        assert torch.equal(want_words, got_words), (n, s0)
    assert reach.count == total


@pytest.mark.gpu
@pytest.mark.parametrize("pair_low", [False, True])
@pytest.mark.parametrize("n", [29, 32, 33, 34])
def test_sweep_marks_equal_the_analytic_fixed_point(n, pair_low):
    """All attractors but one seeded: leaving out (ones, 00) leaves one state unmarked, leaving out (ones, cycle) two.
    With the pair at genes 0, 1 genes 32 and 33 are ring genes, evaluated by the second ballot.  (These marks do not
    depend on how free genes at 32 and above enter the word walk: setting a free ring gene to 0 always stays in the
    basin.  test_copy_network_marks_need_free_upper_genes_both_ways covers that.)"""
    from pbn_rl_b200.discover import ReachMarks
    left = ("ones", "cycle") if pair_low else ("ones", "00")
    seeded = [a for a in ATTRACTORS if a != left]
    env = _env(_trap(n, pair_low))
    try:
        reach = ReachMarks(env)
        seeds = [s for a in seeded for s in trap_attractor_states(n, pair_low, a)]
        assert reach.mark(seeds + [1 << n, (1 << 40) + 1]) == len(seeds)     # states >= 2^N are ignored
        reach.close()
        assert reach.uncovered == len(trap_attractor_states(n, pair_low, left))
        _assert_marks(reach, n, lambda st: trap_reaches(st, n, pair_low, seeded))
        assert reach.unmarked_sample(1024) == trap_attractor_states(n, pair_low, left)[:1]
    finally:
        env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [33, 34])
def test_copy_network_marks_need_free_upper_genes_both_ways(n):
    """copy_network(n): genes n-6..n-1 are free whenever they differ from their sources 0..5, so genes 32 (and 33) are
    free in half of all states.  A state whose gene g >= 32 differs from a seed's, where the seed has g equal to its
    source, is marked only through the successor with the free gene g set to the seed's value: 1 for some seeds, 0 for
    others.  On 12- and 13-gene analogues with the ballot split at gene 10 or 11, these marks tell the correct word walk
    from one that leaves the upper free genes out of H, shifts them one bit short, or takes them as fixed ones."""
    from pbn_rl_b200.discover import ReachMarks
    rng = np.random.default_rng(n)
    seeds = sorted({int(x) for x in rng.integers(0, 1 << n, size=64)})
    need = {((z >> g) & 1) for z in seeds for g in range(32, n) if (z >> g) & 1 == (z >> (g - n + 6)) & 1}
    assert need == {0, 1}                # seeds that gene 32 or 33 must reach by being set to 1, and by being set to 0
    env = _env(_net(copy_network(n)))
    try:
        reach = ReachMarks(env)
        assert reach.mark(seeds) == len(seeds)
        reach.close()
        _assert_marks(reach, n, lambda st: copy_reaches(st, n, seeds))
        assert reach.count > 8 * len(seeds)
    finally:
        env.close()


# ---- 2. the search on trap33 / trap34 -------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("n", [33, 34])
def test_search_finds_what_the_seeding_misses(n):
    """1024 seeding rollouts find the three all-zeros attractors; the sweep leaves the four all-ones states unmarked
    and the discovery round finds the other three."""
    from pbn_rl_b200.discover import find_attractors_exhaustive
    got, info = find_attractors_exhaustive(_trap(n, False), seed_rollouts=1024)
    want = sorted((sorted(trap_attractor_states(n, False, a)) for a in ATTRACTORS), key=lambda m: m[0])
    assert info["states"] == want and len(got) == 6
    assert info["complete"] and info["uncovered"] == 0
    assert info["seeded"] == 3 and info["rounds"] >= 1


# ---- 3. bb33 ---------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_bb33_certified_attractor_table():
    """bb33 is a Boolean network (one predictor per gene): iterating the oracle's update from an attractor's first state
    returns to it after exactly len(attractor) steps, through exactly its states."""
    import json
    from oracle.pbn_oracle import OracleNetwork
    from pbn_rl_b200.discover import find_attractors_exhaustive, find_attractors_rollout
    from pbn_rl_b200.formats import network_from_bnet
    net = network_from_bnet(GOLD / "bb33.bnet")
    got, info = find_attractors_exhaustive(net)
    assert info["complete"] and info["uncovered"] == 0
    _, rinfo = find_attractors_rollout(net)
    assert {tuple(m) for m in rinfo["states"]} <= {tuple(m) for m in info["states"]}
    assert info["seeded"] == len(rinfo["states"])
    assert len(got) == len(info["states"])
    assert sorted(len(m) for m in info["states"]) == [1, 1, 1, 2]         # bb33's certified table: four attractors
    assert [m[0] for m in info["states"]] == sorted(m[0] for m in info["states"])
    want = json.loads((GOLD / "bb33_expected.json").read_text())
    assert net.genes == want["genes"]
    onet = OracleNetwork(want["genes"], [[(e, 1.0)] for e in want["python_exprs"]])
    for members in info["states"]:
        s, seen = members[0], []
        for _ in range(len(members)):
            seen.append(s)
            s = onet.transition(s, 0, [0] * 33, 0)
        assert s == members[0] and sorted(seen) == members


# ---- 4. a random network above 32 genes ------------------------------------------------------------------------------

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


def _successors(onet, s):
    c1, c0 = _descriptor(onet, s)
    free = c1 & c0
    return RO.enumerate_successors(c1 & ~free, free)


@pytest.mark.gpu
def test_random_33_gene_fixed_point_under_the_oracle():
    """make_network(33, 1, 3): one predictor per gene, so every successor set is one state and the attractors are
    short cycles (random networks with two predictors per gene have attractors so large that random seeds mark nearly
    every state).  Seeds are the ends of two-step oracle walks from random states (a uniform state rarely has a
    predecessor), so the walks' earlier states are marked non-seed states.  At sampled states: unmarked => no marked successor, marked and
    not a seed => some marked successor."""
    import torch
    from oracle.pbn_oracle import OracleNetwork
    from pbn_rl_b200.discover import ReachMarks
    n = 33
    spec = make_network(n, 1, 3, seed=33)
    onet = OracleNetwork(*spec)
    rng = np.random.default_rng(33)
    walks = []
    for s in rng.integers(0, 1 << n, size=16):
        path = [int(s)]
        for _ in range(2):
            succ = _successors(onet, path[-1])
            path.append(succ[int(rng.integers(0, len(succ)))])
        walks.append(path)
    seeds = sorted({p[-1] for p in walks})
    env = _env(_net(spec))
    try:
        reach = ReachMarks(env)
        reach.mark(seeds)
        reach.close()
        sample = sorted({int(s) for s in rng.integers(0, 1 << n, size=1024)} | {s for p in walks for s in p})
        succ = [_successors(onet, s) for s in sample]
        flat = torch.tensor([s for s in sample] + [t for ts in succ for t in ts], dtype=torch.int64, device="cuda:0")
        bits = ((reach.marks[flat >> 5].to(torch.int64) >> (flat & 31)) & 1).cpu().numpy().astype(bool)
    finally:
        env.close()
    marked, k = bits[:len(sample)], len(sample)
    n_marked = n_unmarked = 0
    for i, s in enumerate(sample):
        hit = bool(bits[k:k + len(succ[i])].any())
        k += len(succ[i])
        if not marked[i]:
            assert not hit, s
            n_unmarked += 1
        elif s not in seeds:
            assert hit, s
            n_marked += 1
    assert all(marked[sample.index(s)] for p in walks for s in p)
    assert n_marked >= 100 and n_unmarked >= 100          # both sides of the fixed point are sampled


# ---- 5. refusals -----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_35_genes_are_refused():
    import torch
    from pbn_rl_b200._cabi import PBN_ERR_UNSUPPORTED, REACH_MAX_GENES, PbnError
    from pbn_rl_b200.discover import ReachMarks, find_attractors_exhaustive
    assert REACH_MAX_GENES == 34
    net = _trap(35, False)
    env = _env(net)
    try:
        marks = torch.zeros((1 << 10,), dtype=torch.int32, device="cuda:0")
        newly = torch.zeros((1,), dtype=torch.int64, device="cuda:0")
        st = torch.zeros((4,), dtype=torch.int64, device="cuda:0")
        s = env._stream()
        assert env.lib.pbn_reach_sweep(env._h, marks.data_ptr(), newly.data_ptr(), s) == PBN_ERR_UNSUPPORTED
        assert env.lib.pbn_reach_mark(env._h, marks.data_ptr(), st.data_ptr(), 4, newly.data_ptr(), s) == PBN_ERR_UNSUPPORTED
        with pytest.raises(PbnError) as e:
            ReachMarks(env)
        assert e.value.code == PBN_ERR_UNSUPPORTED
    finally:
        env.close()
    with pytest.raises(PbnError) as e:
        find_attractors_exhaustive(net)
    assert e.value.code == PBN_ERR_UNSUPPORTED
    torch.cuda.synchronize()
    assert int(newly.item()) == 0 and int(marks.abs().sum().item()) == 0
