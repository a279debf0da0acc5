"""CPU: the references of the exhaustive attractor search (tests/reach_oracle.py) -- the kernel's split of a successor
set into marks words, and the backward-reachability fixed point against a Tarjan condensation of the STG (K5)."""
import numpy as np
import pytest

import reach_oracle as RO
from helpers import golden, product_net


def test_word_mask_matches_set_enumeration_for_every_low_pattern():
    """All 32 x 32 (fixed low bits, free low genes): the ballot rule gives exactly the low bits of the successors."""
    for fixed in range(32):
        for free in range(32):
            want = 0
            for t in RO.enumerate_successors(fixed, free):
                want |= 1 << (t & 31)
            assert RO.word_mask(fixed, free) == want, (fixed, free)


@pytest.mark.parametrize("n", [3, 5, 6, 12, 23, 28])
def test_successor_words_cover_the_successor_set_exactly(n):
    """The (word, mask) walk of the sweep kernel names every successor once, in 2^|H| distinct words."""
    rng = np.random.default_rng(n)
    for _ in range(200):
        free = 0
        for g in rng.choice(n, size=int(rng.integers(0, min(n, 14) + 1)), replace=False):
            free |= 1 << int(g)
        fixed = int(rng.integers(0, 1 << n)) & ~free
        words = RO.successor_words(fixed, free)
        assert len(words) == 1 << bin(free >> 5).count("1")
        assert len({w for w, _ in words}) == len(words)
        got = sorted(32 * w + b for w, m in words for b in range(32) if (m >> b) & 1)
        assert got == RO.enumerate_successors(fixed, free)
        assert all(t < 1 << n for t in got)


def _condensation_reach(succ):
    """For every state, the set of sink SCCs it reaches, from the strongly connected components of the STG
    (scipy's Tarjan-type algorithm) and a pass over the condensation in reverse topological order."""
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components
    S = len(succ)
    rows = [s for s, ts in enumerate(succ) for _ in ts]
    cols = [t for ts in succ for t in ts]
    k, comp = connected_components(csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(S, S)), directed=True,
                                   connection="strong")
    dag = [set() for _ in range(k)]
    for s, ts in enumerate(succ):
        for t in ts:
            if comp[t] != comp[s]:
                dag[comp[s]].add(comp[t])
    reach = [None] * k
    def visit(c):
        stack = [(c, False)]
        while stack:
            v, done = stack.pop()
            if reach[v] is not None:
                continue
            if done:
                r = {v} if not dag[v] else set()
                for u in dag[v]:
                    r |= reach[u]
                reach[v] = r
            else:
                stack.append((v, True))
                stack.extend((u, False) for u in dag[v] if reach[u] is None)
    for c in range(k):
        visit(c)
    return comp, reach


@pytest.mark.parametrize("name", ["pbn7", "pbn10"])
def test_fixed_point_against_tarjan_condensation(name):
    net = product_net(name)
    succ = RO.successor_lists(net)
    sinks = golden("k5_stg.json")[name]["sink_sccs"]
    every = RO.backward_reach(succ, [s for m in sinks for s in m])
    assert every.all()                          # all sink SCCs as seeds: every state is covered
    comp, reach = _condensation_reach(succ)
    sink_comp = [int(comp[m[0]]) for m in sinks]
    for left_out in range(len(sinks)):
        seeds = [s for a, m in enumerate(sinks) if a != left_out for s in m]
        got = RO.backward_reach(succ, seeds)
        others = {c for a, c in enumerate(sink_comp) if a != left_out}
        want = np.array([bool(reach[comp[s]] & others) for s in range(len(succ))])
        assert np.array_equal(got, want)
        assert not got[sinks[left_out]].any()
        if len(sinks) > 1:
            assert (~got).sum() > 0
        # the unmarked states are closed under successors (they hold the attractor left out)
        for s in np.nonzero(~got)[0]:
            assert not got[succ[s]].any()


def test_pack_marks_layout():
    m = np.zeros(64, dtype=bool)
    m[[0, 31, 32, 63]] = True
    assert RO.pack_marks(m).tolist() == [0x80000001, 0x80000001]
    assert RO.pack_marks(np.array([False, True, False, True, True, False, False, False])).tolist() == [0b11010]
