"""Dense numpy references of exact state distributions (pbn_dp_push, pbn_rl_b200/steady_state.py) for small networks,
built on control_oracle.transition_matrix (the step contract, perturbation masks enumerated explicitly):

- the forward step x P, and the closed loop x M_mu P (flips s -> s ^ mu(s) first);
- the stationary vector pi = pi P from a linear solve (one equation replaced by sum pi = 1), and power iteration;
- marginals and projections of a distribution by explicit loops over the states.
Test infrastructure only; N <= 12.  point_row gives one row of P at any N <= 28 from the successor enumeration."""
import numpy as np

import control_oracle as CO


def dense_transition(onet, mode="none", p=0.0):
    """P of one uncontrolled step: control_oracle.transition_matrix up to 8 genes; above, its algebra as dense
    products, F K_p (model B: the update, then ^ m) and c F + K_p - c I (model A), with K_p[u, t] = p^|u^t|
    (1-p)^(N-|u^t|) from the enumerated mask probabilities (the row-by-row loops cost O(4^N) in Python)."""
    n = CO.n_genes(onet)
    if n <= 8 or CO.MODES[mode] == CO.O.PERT_NONE or p == 0.0:
        return CO.transition_matrix(onet, mode, p)
    S = 1 << n
    f = CO.selection_matrix(onet)
    idx = np.arange(S)
    kp = CO.mask_probabilities(n, p)[idx[:, None] ^ idx[None, :]]
    if CO.MODES[mode] == CO.O.PERT_B:
        return f @ kp
    c = (1.0 - p) ** n
    return c * f + kp - c * np.eye(S)


def closed_loop_matrix(onet, mode="none", p=0.0, masks=None, P=None):
    """P_mu = M_mu P, M_mu[s, s ^ mu(s)] = 1: row s of P_mu is row s ^ mu(s) of P (P itself without masks)."""
    P = dense_transition(onet, mode, p) if P is None else P
    if masks is None:
        return P
    S = P.shape[0]
    return P[np.arange(S) ^ np.asarray(masks, dtype=np.int64)]


def push(onet, x, mode="none", p=0.0, masks=None, P=None):
    """y = x P_mu."""
    return np.asarray(x, dtype=np.float64) @ closed_loop_matrix(onet, mode, p, masks, P)


def stationary(P):
    """pi with pi P = pi, sum pi = 1 (unique for an irreducible chain): (P^T - I) pi = 0 with its last equation
    replaced by the normalisation."""
    S = P.shape[0]
    a = P.T - np.eye(S)
    a[-1, :] = 1.0
    b = np.zeros(S)
    b[-1] = 1.0
    return np.linalg.solve(a, b)


def power_iteration(P, tol=1e-13, max_iters=1 << 20, x=None):
    """x <- x P from ``x`` (default uniform) until |x P - x|_1 < tol; returns (x, iterations)."""
    S = P.shape[0]
    x = np.full(S, 1.0 / S) if x is None else np.asarray(x, dtype=np.float64)
    for it in range(1, max_iters + 1):
        y = x @ P
        y /= y.sum()
        if np.abs(y - x).sum() < tol:
            return y, it
        x = y
    return x, max_iters


def marginals(x):
    """P(gene g = 1) by a loop over the states."""
    x = np.asarray(x, dtype=np.float64)
    n = x.size.bit_length() - 1
    out = np.zeros(n)
    for s in range(x.size):
        for g in range(n):
            if (s >> g) & 1:
                out[g] += x[s]
    return out


def projection(x, genes):
    """The distribution of the states projected onto ``genes`` (bin bit j = gene genes[j]) by a loop over the states."""
    x = np.asarray(x, dtype=np.float64)
    out = np.zeros(1 << len(genes))
    for s in range(x.size):
        b = sum(((s >> g) & 1) << j for j, g in enumerate(genes))
        out[b] += x[s]
    return out


def point_row(net, s):
    """(successor indices, weights) of state s under the selection step (p = 0): row s of F, for N <= 28, from the
    successor-set enumeration of control_oracle (the lowest free gene is the lowest bit of the enumeration order)."""
    q1, q0 = CO.gene_split(net, [s])
    n = CO.n_genes(net)
    free = [i for i in range(n) if q1[0, i] > 0.0 and q0[0, i] > 0.0]
    fixed = sum(1 << i for i in range(n) if q0[0, i] == 0.0)
    return CO._successors(free, q1[0], q0[0], fixed)
