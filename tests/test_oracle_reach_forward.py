"""CPU: the references of the forward closure over the state bitset (tests/reach_forward_oracle.py) -- the numpy fixed
point against a breadth-first search, the kernel's word walk against set enumeration for every state, and the closed
forms of the networks the GPU tests build."""
import numpy as np
import pytest

import reach_forward_oracle as RF
import reach_oracle as RO
from helpers import make_network, product_net

NETS = {"n3": (3, 2, 2, 3), "n4": (4, 2, 3, 4), "n5": (5, 2, 2, 5), "n9": (9, 2, 3, 9), "n12": (12, 3, 2, 13)}


def _net(spec):
    from pbn_rl_b200 import PBNNetwork
    return PBNNetwork.from_expressions(*spec)


def _made(name):
    if name in ("pbn7", "pbn10"):
        return product_net(name)
    return _net(make_network(*NETS[name][:3], seed=NETS[name][3]))


def _sink_sccs(succ):
    from pbn_rl_b200.discover import sink_sccs_of_closed_set
    return sink_sccs_of_closed_set({s: list(ts) for s, ts in enumerate(succ)})


@pytest.mark.parametrize("n", range(3, 13))
def test_forward_reach_equals_bfs(n):
    succ = RO.successor_lists(_net(make_network(n, 2, 3, seed=100 + n)))
    rng = np.random.default_rng(n)
    for seeds in ([0], [(1 << n) - 1], [int(x) for x in rng.integers(0, 1 << n, size=3)],
                  [int(x) for x in rng.integers(0, 1 << n, size=max(1, (1 << n) // 16))]):
        assert np.array_equal(RF.forward_reach(succ, seeds), RF.forward_reach_bfs(succ, seeds)), (n, seeds[:3])


@pytest.mark.parametrize("name", ["n3", "n4", "n5", "n9", "n12", "pbn7", "pbn10"])
def test_forward_word_walk_sets_exactly_the_successors(name):
    """For every state: the words base | c under the mask M name exactly the successor set, and no state >= 2^N (at
    N < 5 the mask stays inside the partial word)."""
    from pbn_rl_b200.attractors import _successor_sets
    net = _made(name)
    n = net.n_genes
    can1, can0 = _successor_sets(net)
    for s in range(1 << n):
        c1, c0 = int(can1[s]), int(can0[s])
        free = c1 & c0
        got = RF.forward_word_walk(c1 & ~free, free)
        assert got == RO.enumerate_successors(c1 & ~free, free), (name, s)
        assert all(t < 1 << n for t in got)


@pytest.mark.parametrize("n,free", [(6, [0, 1]), (8, [0, 1, 2]), (9, [1, 4, 6, 7]), (10, [5, 6, 8, 9]), (7, [0, 1, 2, 3, 4, 5])])
def test_free_block_closed_form(n, free):
    from pbn_rl_b200.attractors import _successor_sets
    net = _net(RF.free_block_network(n, free))
    assert _sink_sccs(RO.successor_lists(net)) == [a.tolist() for a in RF.free_block_attractors(n, free)]
    can1, can0 = _successor_sets(net)
    assert all(int(c1) & int(c0) == sum(1 << g for g in free) for c1, c0 in zip(can1, can0))   # free in every state


@pytest.mark.parametrize("n,f", [(6, 3), (8, 5), (9, 4), (11, 7)])
def test_gated_trap_closed_form(n, f):
    net = _net(RF.gated_trap_network(n, f))
    succ = RO.successor_lists(net)
    (big, smallest), small = RF.gated_trap_attractors(n, f)
    sinks = _sink_sccs(succ)
    assert sorted(sinks, key=len)[-1][0] == smallest and len(sorted(sinks, key=len)[-1]) == big
    assert sorted(m for m in sinks if len(m) < big) == small
    hidden = small[1][0]
    basin = RO.backward_reach(succ, [hidden])
    assert int(basin.sum()) == 1 << (n - f - 1)           # the gate off, the ring all ones, any copy genes
