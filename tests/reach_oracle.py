"""Host references for the exhaustive attractor search (pbn_reach_mark / pbn_reach_sweep, csrc/discover.cuh).

* :func:`successor_lists` -- the perturbation-free STG as explicit successor lists (attractors._successor_sets /
  _successors), N <= 12.
* :func:`backward_reach` -- the sweep's fixed point restated: every state that reaches a seed, by breadth-first search
  over the reversed edges.
* :func:`word_mask` / :func:`successor_words` -- the kernel's split of a successor set into marks words (the high free
  genes pick the word, the low ones a mask inside it), restated bit for bit.
* :func:`pack_marks` -- a boolean state vector in the marks layout (bit s & 31 of word s >> 5).
"""
import numpy as np


def successor_lists(net):
    from pbn_rl_b200.attractors import _successor_sets, _successors
    n = net.n_genes
    assert n <= 12
    can1, can0 = _successor_sets(net)
    return [_successors(s, int(can1[s]), int(can0[s]), n) for s in range(1 << n)]


def backward_reach(succ, seeds):
    """bool [2^N]: the states from which some seed is reachable (the seeds included)."""
    pred = [[] for _ in succ]
    for s, ts in enumerate(succ):
        for t in ts:
            pred[t].append(s)
    out = np.zeros(len(succ), dtype=bool)
    todo = [int(s) for s in seeds if 0 <= int(s) < len(succ)]
    out[todo] = True
    while todo:
        for q in pred[todo.pop()]:
            if not out[q]:
                out[q] = True
                todo.append(q)
    return out


def pack_marks(marked):
    """bool [2^N] -> uint32 [max(1, 2^N / 32)] words, bit s & 31 of word s >> 5."""
    marked = np.asarray(marked, dtype=bool)
    words = np.zeros(max(1, (len(marked) + 31) // 32), dtype=np.uint32)
    for s in np.nonzero(marked)[0]:
        words[s >> 5] |= np.uint32(1 << (int(s) & 31))
    return words


def word_mask(fixed, free):
    """The kernel's word-local mask: bit b set iff (b ^ fixed) & 31 & ~free == 0."""
    return sum(1 << b for b in range(32) if ((b ^ fixed) & 31 & ~free) == 0)


def successor_words(fixed, free):
    """(word, mask) pairs the kernel tests for a state with these fixed / free genes, in its order: lane l takes the
    subset of the five lowest high free genes (genes >= 5) given by the bits of l, the remaining high genes advance by
    c -> (c - H) & H."""
    m = word_mask(fixed, free)
    base, hw = fixed >> 5, free >> 5
    hhi, low_genes = hw, []
    while hhi and len(low_genes) < 5:
        g = hhi & -hhi
        hhi ^= g
        low_genes.append(g)
    out = []
    chi = 0
    while True:
        for lane in range(1 << len(low_genes)):
            clo = sum(g for j, g in enumerate(low_genes) if (lane >> j) & 1)
            out.append((base | clo | chi, m))
        chi = (chi - hhi) & hhi
        if chi == 0:
            return out


def enumerate_successors(fixed, free):
    """The successor set {fixed & ~free | c : c subset of free}, by set enumeration."""
    out = [fixed & ~free]
    b = free
    while b:
        low = b & -b
        out += [t | low for t in out]
        b ^= low
    return sorted(out)
