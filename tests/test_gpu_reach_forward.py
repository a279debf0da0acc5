"""GPU: the forward closure over the state bitset (pbn_reach_forward) and the exhaustive search with closure="bitset".

The forward sweeps' fixed point is checked bit for bit against the numpy restatement (tests/reach_forward_oracle.py);
the search against closed-form attractors of free-block networks (attractors of 2^f states, f free genes in each of
their states, beyond the hash closure's limits), against the hash closure where both complete, and against the host
Tarjan up to 16 genes."""
import numpy as np
import pytest

import reach_forward_oracle as RF
import reach_oracle as RO
from helpers import GOLD, golden, make_network, product_net

pytestmark = pytest.mark.gpu

MADE = {  # name -> make_network(n, kmax, amax, seed), as in test_gpu_reach.py
    "n3": (3, 2, 2, 3), "n5": (5, 2, 2, 5), "n6": (6, 2, 2, 7), "n9": (9, 2, 3, 9), "n12": (12, 3, 2, 13),
    "wide12": (12, 3, 12, 7), "n16": (16, 2, 4, 1), "n20": (20, 2, 3, 21), "n24": (24, 2, 3, 25),
    "dense20": (20, 3, 4, 20),
}


def trap_network(n):
    """As in test_gpu_reach.py: six attractors, three of them with basins of one or two states."""
    k = n - 2
    genes = ["x%d" % i for i in range(n)]
    exprs = [[("( x%d & x%d )" % (i, (i + 1) % k), 0.5), ("( x%d & x%d )" % (i, (i - 1) % k), 0.5)] for i in range(k)]
    exprs += [[("x%d" % (n - 1), 1.0)], [("x%d" % (n - 2), 1.0)]]
    return genes, exprs


def _net(name):
    from pbn_rl_b200 import PBNNetwork
    from pbn_rl_b200.formats import network_from_bnet
    if name in ("pbn7", "pbn10", "pbn28"):
        return product_net(name)
    if name == "bb33":
        return network_from_bnet(GOLD / "bb33.bnet")
    if name.startswith("trap"):
        return PBNNetwork.from_expressions(*trap_network(int(name[4:])))
    spec = MADE[name]
    return PBNNetwork.from_expressions(*make_network(spec[0], spec[1], spec[2], seed=spec[3]))


def _spec_net(genes_exprs):
    from pbn_rl_b200 import PBNNetwork
    return PBNNetwork.from_expressions(*genes_exprs)


def _env(net):
    from pbn_rl_b200 import VecPBNEnv
    return VecPBNEnv(net, 1024, None, device="cuda:0", horizon=0, bins=1, perturb_p=0.0)


# ---- 1. forward sweeps against the oracle, bit for bit --------------------------------------------------------------

@pytest.mark.parametrize("name", ["pbn7", "pbn10", "n3", "n5", "n6", "n9", "n12", "wide12"])
def test_forward_fixed_point_equals_oracle(name):
    import torch
    from pbn_rl_b200.discover import _ForwardWorkspace
    net = _net(name)
    n, S = net.n_genes, 1 << net.n_genes
    succ = RO.successor_lists(net)
    rng = np.random.default_rng(n)
    seed_sets = [[0], [S - 1], [int(x) for x in rng.integers(0, S, size=3)],
                 [int(x) for x in rng.integers(0, S, size=max(1, S // 16))]]
    env = _env(net)
    try:
        ws = _ForwardWorkspace(env)
        lib, h, st = env.lib, env._h, env._stream()
        for seeds in seed_sets:
            ws.set.zero_()
            ws.done.zero_()
            for s in seeds:
                ws._mark(ws.set, s)
            reached = expanded = 0
            while True:
                ws.newly.zero_()
                assert lib.pbn_reach_forward(h, ws.set.data_ptr(), ws.done.data_ptr(), ws.newly.data_ptr(), st) == 0
                r, e = ws.newly.tolist()
                reached, expanded = reached + r, expanded + e
                if e == 0:
                    break
            want = RF.forward_reach(succ, seeds)
            got = ws.set.cpu().numpy().view(np.uint32)
            assert np.array_equal(got, RO.pack_marks(want)), (name, seeds[:4])       # all 2^N bits, partial word too
            assert torch.equal(ws.set, ws.done)
            assert expanded == int(want.sum()) == reached + len(set(seeds))
    finally:
        env.close()


# ---- 2. free-block networks, closed form ----------------------------------------------------------------------------

def _assert_free_block(info, n, free):
    want = [a.tolist() for a in RF.free_block_attractors(n, free)]
    assert info["states"] == want
    assert info["complete"] and info["uncovered"] == 0 and info["oversized"] == []


def test_free_block_beyond_the_hash_closure_at_20_genes():
    """18 free genes: the hash closure refuses every attractor state (more than 16 free genes); the bitset closure
    lists both attractors."""
    from pbn_rl_b200.discover import find_attractors_exhaustive
    free = list(range(18))
    net = _spec_net(RF.free_block_network(20, free))
    _, hinfo = find_attractors_exhaustive(net, max_attractor_states=1 << 18)
    assert not hinfo["complete"] and hinfo["uncovered"] > 0 and "oversized" not in hinfo
    _, info = find_attractors_exhaustive(net, max_attractor_states=1 << 18, closure="bitset")
    _assert_free_block(info, 20, free)


@pytest.mark.parametrize("free", [list(range(18)), list(range(16)) + [32, 33]], ids=["low", "upper"])
def test_free_block_at_34_genes(free):
    """The "upper" block makes genes 32 and 33 free: the wide instance walks its upper H bits."""
    from pbn_rl_b200.discover import find_attractors_exhaustive
    got, info = find_attractors_exhaustive(_spec_net(RF.free_block_network(34, free)), max_attractor_states=1 << 18,
                                           closure="bitset")
    _assert_free_block(info, 34, free)
    assert len(got) == 2


def test_free_block_oversized_at_34_genes():
    """22 free genes, beyond even the hash kernel's cap of 20: every state is marked, and the two attractors of 2^22
    states are reported, not listed."""
    from pbn_rl_b200.discover import find_attractors_exhaustive
    _, info = find_attractors_exhaustive(_spec_net(RF.free_block_network(34, list(range(22)))), closure="bitset")
    assert info["uncovered"] == 0 and not info["complete"] and info["states"] == []
    assert info["oversized"] == [(1 << 22, 0), (1 << 22, ((1 << 12) - 1) << 22)]


# ---- 3. dense20 ---------------------------------------------------------------------------------------------------

def test_dense20():
    from pbn_rl_b200.discover import find_attractors_exhaustive
    net = _net("dense20")
    _, hinfo = find_attractors_exhaustive(net, max_attractor_states=1 << 20)
    _, binfo = find_attractors_exhaustive(net, max_attractor_states=1 << 20, closure="bitset")
    assert hinfo["complete"] and binfo["complete"] and binfo["uncovered"] == 0
    assert binfo["states"] == hinfo["states"]
    _, info = find_attractors_exhaustive(net, closure="bitset")
    assert info["uncovered"] == 0 and not info["complete"]
    big = [m for m in hinfo["states"] if len(m) > 1 << 14]
    assert len(big) == 1 and len(big[0]) == 458752
    assert info["oversized"] == [(458752, big[0][0])]
    assert info["states"] == [m for m in hinfo["states"] if len(m) <= 1 << 14]


# ---- 4. the same tables where both closures complete ----------------------------------------------------------------

@pytest.mark.parametrize("name", ["n16", "n20", "n24", "pbn28", "trap34", "bb33"])
def test_bitset_equals_hash(name):
    from pbn_rl_b200.discover import find_attractors_exhaustive
    net = _net(name)
    _, hinfo = find_attractors_exhaustive(net)
    _, binfo = find_attractors_exhaustive(net, closure="bitset")
    assert hinfo["complete"] and binfo["complete"] and binfo["uncovered"] == 0 and binfo["oversized"] == []
    assert binfo["states"] == hinfo["states"] and binfo["seeded"] == hinfo["seeded"]


@pytest.mark.parametrize("seed_rollouts", [0, 1 << 16])
@pytest.mark.parametrize("name", ["pbn7", "pbn10", "n12", "n16", "trap12", "trap16"])
def test_bitset_equals_tarjan(name, seed_rollouts):
    from pbn_rl_b200 import find_attractors_stg
    from pbn_rl_b200.discover import find_attractors_exhaustive
    net = _net(name)
    want, winfo = find_attractors_stg(net)
    got, info = find_attractors_exhaustive(net, seed_rollouts=seed_rollouts, closure="bitset")
    assert info["states"] == winfo["sink_sccs"] and got.attractors == want.attractors
    assert info["complete"] and info["uncovered"] == 0 and info["oversized"] == []
    if seed_rollouts == 0:
        assert info["seeded"] == 0 and info["rounds"] >= 1 and info["closures"] >= len(info["states"])


# ---- 5. the restart path --------------------------------------------------------------------------------------------

def test_restart_from_a_transient_state_with_several_attractors_downstream():
    """A pbn10 state whose forward closure holds several sink SCCs, with no rollout before the call: the first closure
    is not strongly connected, the search restarts inside it and returns one of the STG's sink SCCs -- the same one
    on a second call."""
    from pbn_rl_b200.discover import _ForwardWorkspace, attractor_in_closure
    net = _net("pbn10")
    sinks = [sorted(m) for m in golden("k5_stg.json")["pbn10"]["sink_sccs"]]
    succ = RO.successor_lists(net)
    fw = [RF.forward_reach(succ, [s]) for s in range(1 << 10)]
    holds = [sum(bool(fw[s][m[0]]) for m in sinks) for s in range(1 << 10)]
    s = int(np.argmax(holds))
    assert holds[s] >= 2
    env = _env(net)
    try:
        out = []
        for _ in range(2):
            ws = _ForwardWorkspace(env)
            size, members = attractor_in_closure(env, s, burn_in=0, ws=ws)
            assert ws.closures >= 2                                        # it did restart
            out.append(members)
            assert size == len(members)
        assert out[0] in sinks and out[0] == out[1] and fw[s][out[0][0]]
        size, members, bits = attractor_in_closure(env, s, max_states=len(out[0]) - 1, burn_in=0, return_bits=True)
        assert members is None and size == len(out[0])
        assert np.array_equal(bits.cpu().numpy().view(np.uint32), RO.pack_marks(np.isin(np.arange(1 << 10), out[0])))
        assert attractor_in_closure(env, s)[1] in sinks                  # restarts after rollouts (burn_in=64)
    finally:
        env.close()


# ---- 6. an oversized attractor does not hide the others --------------------------------------------------------------

def test_oversized_attractor_does_not_hide_the_others():
    """gated_trap_network(20, 18): an attractor of 2^18 states (18 free genes), the state 0, and a fixed point whose
    basin is 2 states.  The bitset closure marks the big one, reports it, and lists both fixed points; the hash
    closure fails on the big one and never reaches the small basin."""
    from pbn_rl_b200.discover import find_attractors_exhaustive
    n, f = 20, 18
    net = _spec_net(RF.gated_trap_network(n, f))
    (big, smallest), small = RF.gated_trap_attractors(n, f)
    _, info = find_attractors_exhaustive(net, closure="bitset")
    assert info["states"] == small and info["oversized"] == [(big, smallest)]
    assert info["uncovered"] == 0 and not info["complete"]
    _, hinfo = find_attractors_exhaustive(net)
    assert not hinfo["complete"] and hinfo["uncovered"] > 0
    assert hinfo["states"] != small and all(m in small for m in hinfo["states"])


# ---- 7. refusals ---------------------------------------------------------------------------------------------------

def test_refusals():
    import torch
    from pbn_rl_b200._cabi import PBN_ERR_INVALID, PBN_ERR_UNSUPPORTED, PbnError
    from pbn_rl_b200.discover import attractor_in_closure, find_attractors_exhaustive
    marks = torch.zeros((1 << 10,), dtype=torch.int32, device="cuda:0")
    done = torch.zeros_like(marks)
    newly = torch.zeros((2,), dtype=torch.int64, device="cuda:0")
    big = _env(_spec_net(trap_network(35)))
    try:
        assert big.lib.pbn_reach_forward(big._h, marks.data_ptr(), done.data_ptr(), newly.data_ptr(),
                                         big._stream()) == PBN_ERR_UNSUPPORTED
        with pytest.raises(PbnError) as e:
            attractor_in_closure(big, 0)
        assert e.value.code == PBN_ERR_UNSUPPORTED
    finally:
        big.close()
    with pytest.raises(ValueError):
        find_attractors_exhaustive(_net("pbn10"), closure="list")
    env = _env(_net("pbn10"))
    try:
        h, s, lib = env._h, env._stream(), env.lib
        assert lib.pbn_reach_forward(h, None, done.data_ptr(), newly.data_ptr(), s) == PBN_ERR_INVALID
        assert lib.pbn_reach_forward(h, marks.data_ptr(), None, newly.data_ptr(), s) == PBN_ERR_INVALID
        assert lib.pbn_reach_forward(h, marks.data_ptr(), done.data_ptr(), None, s) == PBN_ERR_INVALID
        assert lib.pbn_reach_forward(None, marks.data_ptr(), done.data_ptr(), newly.data_ptr(), s) == PBN_ERR_INVALID
        torch.cuda.synchronize()
        assert int(newly.abs().sum().item()) == 0 and int(marks.abs().sum().item()) == 0
    finally:
        env.close()
