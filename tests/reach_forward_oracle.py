"""Host references for the forward closure over the state bitset (pbn_reach_forward, discover.attractor_in_closure).

* :func:`forward_reach` -- the forward sweeps' fixed point restated: every state reachable from a seed, by repeated
  numpy edge relaxation over the dense successor lists of reach_oracle.successor_lists.
* :func:`forward_reach_bfs` -- the same set by a plain breadth-first search, the brute force the first is checked against.
* :func:`forward_word_walk` -- the kernel's expansion of one state restated bit for bit: the words ``base | c`` for the
  subsets ``c`` of the high free genes, each OR-ed with the word-local mask ``M``.
* :func:`free_block_network` / :func:`gated_trap_network` -- networks whose attractors are known in closed form, with
  attractors of 2^f states (f free genes in every state of them).
"""
import numpy as np

import reach_oracle as RO


def forward_reach(succ, seeds):
    """bool [2^N]: the states reachable from some seed (the seeds included)."""
    src = np.array([s for s, ts in enumerate(succ) for _ in ts], dtype=np.int64)
    dst = np.array([t for ts in succ for t in ts], dtype=np.int64)
    out = np.zeros(len(succ), dtype=bool)
    out[[int(s) for s in seeds if 0 <= int(s) < len(succ)]] = True
    while True:
        nxt = out.copy()
        nxt[dst[out[src]]] = True
        if np.array_equal(nxt, out):
            return out
        out = nxt


def forward_reach_bfs(succ, seeds):
    out = np.zeros(len(succ), dtype=bool)
    todo = [int(s) for s in seeds if 0 <= int(s) < len(succ)]
    out[todo] = True
    while todo:
        for t in succ[todo.pop()]:
            if not out[t]:
                out[t] = True
                todo.append(t)
    return out


def forward_word_walk(fixed, free):
    """The states the forward kernel sets for one state with these fixed / free genes: for every (word, M) of the walk
    (reach_oracle.successor_words, lane for lane), the bits of M in that word."""
    return sorted(32 * w + b for w, m in RO.successor_words(fixed, free) for b in range(32) if (m >> b) & 1)


def free_block_network(n, free):
    """Genes in ``free`` have the predictors x_i and ~x_i, so they are free in every state.  The lowest other gene (the
    key) keeps its value and the remaining genes copy it.  Two attractors, of 2^len(free) states each: the free genes
    arbitrary and the other genes all 0 or all 1."""
    free = sorted(free)
    rest = [g for g in range(n) if g not in free]
    key = rest[0]
    genes = ["x%d" % i for i in range(n)]
    exprs = []
    for i in range(n):
        if i in free:
            exprs.append([("x%d" % i, 0.5), ("~ x%d" % i, 0.5)])
        else:
            exprs.append([("x%d" % key, 1.0)])
    return genes, exprs


def free_block_attractors(n, free):
    """The two attractors of free_block_network(n, free) as sorted int64 arrays."""
    free = sorted(free)
    x = np.arange(1 << len(free), dtype=np.int64)
    low = np.zeros_like(x)
    for j, g in enumerate(free):
        low |= ((x >> j) & 1) << g
    high = ((1 << n) - 1) & ~sum(1 << g for g in free)
    return [np.sort(low), np.sort(low | high)]


def gated_trap_network(n, f):
    """Gene 0 (the gate) keeps its value, genes 1..n-f-1 copy it, genes n-f..n-1 form a ring.  Gate on: every ring gene
    has the predictors x_i and ~x_i (free).  Gate off: ring gene i keeps x_i & x_(i+1) or x_i & x_(i-1), so a zero
    spreads and 'all ones' is reached only from itself.  Three attractors: the gate and its copies on with the ring
    arbitrary (2^f states, smallest state 2^(n-f) - 1), the state 0, and the ring all ones with everything else off
    (its basin: those states with any copy genes, 2^(n-f-1) states)."""
    c0 = n - f
    genes = ["x%d" % i for i in range(n)]
    exprs = [[("x0", 1.0)]] + [[("x0", 1.0)] for _ in range(1, c0)]
    for j in range(f):
        g, nx, pv = c0 + j, c0 + (j + 1) % f, c0 + (j - 1) % f
        exprs.append([("( x0 & x%d ) | ( ~ x0 & x%d & x%d )" % (g, g, nx), 0.5),
                      ("( x0 & ~ x%d ) | ( ~ x0 & x%d & x%d )" % (g, g, pv), 0.5)])
    return genes, exprs


def gated_trap_attractors(n, f):
    """(big attractor's size and smallest state, the sorted small attractors) of gated_trap_network(n, f)."""
    c0 = n - f
    return (1 << f, (1 << c0) - 1), [[0], [((1 << f) - 1) << c0]]
