"""Dense numpy restatement of exact finite-horizon PBN control (include/pbn_b200.h, "Exact optimal control";
pbn_rl_b200/control.py) for small networks, written from the step contract rather than from the kernels:

- the selection step F in its per-gene product form (gene i goes to 1 with probability q_i(u) = sum of the selection
  probabilities of its predictors that yield 1), evaluated with the oracle network's expressions;
- perturbation by explicit enumeration of the perturbation masks and their probabilities p^|m| (1-p)^(N-|m|) (model A:
  a perturbed step skips the update and lands on u ^ m; model B: the update, then ^ m), not through butterflies;
- the maximum over flip sets by brute-force enumeration of every allowed mask with the contract's tie order (fewer
  flips, then larger w[s ^ m], then smaller s ^ m);
- the finite-horizon recursion of both objectives ("return", "steps").
Test infrastructure only; N <= 12 for the dense forms.  The sampled forms scale to N = 28: sparse_expect enumerates
a state's successor set in chunks and gathers u through a formula (u_hash, w_ties, w_rounding) where no 2^N vector
is wanted, kp_tensor applies the perturbation channel gene by gene (N <= 24), and improve_brute_states /
classify_states evaluate the brute force and the classification at listed states only.
"""
import itertools

import numpy as np

from oracle import pbn_oracle as O

MODES = {"none": O.PERT_NONE, "A": O.PERT_A, "B": O.PERT_B}


def n_genes(net):
    return net.n if hasattr(net, "np_code") else net.n_genes


def gene_probabilities(net, states=None):
    """q[x, i] = probability that gene i is 1 after the selection step from state x (all 2^N states by default).
    ``net``: an oracle network (its expressions are evaluated) or a PBNNetwork (its truth tables are looked up)."""
    n = n_genes(net)
    xs = np.arange(1 << n, dtype=np.int64) if states is None else np.asarray(states, dtype=np.int64)
    q = np.zeros((xs.size, n), dtype=np.float64)
    if hasattr(net, "np_code"):
        ns = {g: ((xs >> i) & 1).astype(bool) for i, g in enumerate(net.genes)}
        for i in range(n):
            for code, p in zip(net.np_code[i], net.probs[i]):
                v = np.broadcast_to(np.asarray(eval(code, {}, ns), dtype=bool), xs.shape)
                q[:, i] += p * v
        return q
    for i, (fs, ps) in enumerate(zip(net.functions, net.probabilities)):
        for f, p in zip(fs, ps):
            idx = np.zeros(xs.size, dtype=np.int64)
            for j, g in enumerate(f.inputs):
                idx |= ((xs >> g) & 1) << j
            tab = np.array([(f.lut >> a) & 1 for a in range(1 << f.arity)], dtype=bool)
            q[:, i] += p * tab[idx]
    return q


def selection_matrix(onet):
    """F[x, t] = prod_i (q_i(x) if t_i else 1 - q_i(x))   (dense, N <= 12)."""
    n = n_genes(onet)
    q = gene_probabilities(onet)
    t = np.arange(1 << n, dtype=np.int64)
    f = np.ones((1 << n, 1 << n), dtype=np.float64)
    for i in range(n):
        bit = ((t >> i) & 1).astype(bool)
        f *= np.where(bit[None, :], q[:, i:i + 1], 1.0 - q[:, i:i + 1])
    return f


def mask_probabilities(n, p):
    """pm[m] = p^|m| (1 - p)^(N - |m|) for every perturbation mask m."""
    pc = np.array([bin(m).count("1") for m in range(1 << n)])
    return (p ** pc) * ((1.0 - p) ** (n - pc))


def transition_matrix(onet, mode="none", p=0.0):
    """P[u, t] of one uncontrolled step, built row by row: selection, then every perturbation mask enumerated."""
    n = n_genes(onet)
    S = 1 << n
    f = selection_matrix(onet)
    if MODES[mode] == O.PERT_NONE or p == 0.0:
        return f
    pm = mask_probabilities(n, p)
    idx = np.arange(S)
    out = np.zeros_like(f)
    for u in range(S):
        if MODES[mode] == O.PERT_A:
            out[u] += pm[0] * f[u]
            for m in range(1, S):
                out[u, u ^ m] += pm[m]
        else:
            for m in range(S):
                out[u, idx ^ m] += pm[m] * f[u]
    return out


def expect(onet, u, mode="none", p=0.0, f=None):
    """(P u) for all states without building P: F u, with the perturbation masks enumerated explicitly."""
    n = n_genes(onet)
    S = 1 << n
    f = selection_matrix(onet) if f is None else f
    u = np.asarray(u, dtype=np.float64)
    if MODES[mode] == O.PERT_NONE or p == 0.0:
        return f @ u
    pm = mask_probabilities(n, p)
    idx = np.arange(S)
    if MODES[mode] == O.PERT_A:
        out = pm[0] * (f @ u)
        for m in range(1, S):
            out += pm[m] * u[idx ^ m]
        return out
    ku = np.zeros(S)
    for m in range(S):
        ku += pm[m] * u[idx ^ m]
    return f @ ku


def gene_split(net, states):
    """(q1, q0) [len(states), N]: the summed selection probabilities of gene i's predictors that yield 1 / yield 0 in
    each listed state.  Gene i is free where both are > 0, fixed to 1 where q0 = 0 and fixed to 0 where q1 = 0."""
    n = n_genes(net)
    xs = np.asarray(states, dtype=np.int64)
    q1 = np.zeros((xs.size, n), dtype=np.float64)
    q0 = np.zeros((xs.size, n), dtype=np.float64)
    if hasattr(net, "np_code"):
        ns = {g: ((xs >> i) & 1).astype(bool) for i, g in enumerate(net.genes)}
        for i in range(n):
            for code, p in zip(net.np_code[i], net.probs[i]):
                v = np.broadcast_to(np.asarray(eval(code, {}, ns), dtype=bool), xs.shape)
                q1[:, i] += np.where(v, p, 0.0)
                q0[:, i] += np.where(v, 0.0, p)
        return q1, q0
    for i, (fs, ps) in enumerate(zip(net.functions, net.probabilities)):
        for f, p in zip(fs, ps):
            idx = np.zeros(xs.size, dtype=np.int64)
            for j, g in enumerate(f.inputs):
                idx |= ((xs >> g) & 1) << j
            tab = np.array([(f.lut >> a) & 1 for a in range(1 << f.arity)], dtype=bool)
            v = tab[idx]
            q1[:, i] += np.where(v, p, 0.0)
            q0[:, i] += np.where(v, 0.0, p)
    return q1, q0


def free_counts(net, states):
    """Number of free genes (predictors yielding both values) of each listed state: log2 of its successor count."""
    q1, q0 = gene_split(net, states)
    return ((q1 > 0.0) & (q0 > 0.0)).sum(axis=1)


def _gather(u, idx):
    return u(idx) if callable(u) else np.asarray(u, dtype=np.float64)[idx]


def _successors(genes, q1, q0, base):
    """Indices and weights of every assignment of ``genes`` (lowest gene = lowest bit of the enumeration order)."""
    t = np.full(1, base, dtype=np.int64)
    wt = np.ones(1)
    for i in genes:
        t = np.concatenate([t, t | (1 << int(i))])
        wt = np.concatenate([wt * q0[i], wt * q1[i]])
    return t, wt


def sparse_expect(onet, u, states, chunk_bits=20):
    """(F u)(x) for the listed states by enumerating each state's successor set (p = 0).  ``u``: an array over all
    states or a callable ``u(indices int64) -> float64``, so that nothing of size 2^N is built.  The lowest
    ``chunk_bits`` free genes of a state are enumerated as one vector of at most 2^chunk_bits successors; the higher
    free genes run in an outer loop, so a state of 28 free genes is 2^(28 - chunk_bits) gathers of 2^chunk_bits."""
    q1, q0 = gene_split(onet, states)
    n = n_genes(onet)
    out = np.zeros(len(states))
    for r in range(len(states)):
        free = [i for i in range(n) if q1[r, i] > 0.0 and q0[r, i] > 0.0]
        fixed = sum(1 << i for i in range(n) if q0[r, i] == 0.0)
        lo, hi = free[:chunk_bits], free[chunk_bits:]
        t_lo, w_lo = _successors(lo, q1[r], q0[r], fixed)
        t_hi, w_hi = _successors(hi, q1[r], q0[r], 0)
        acc = 0.0
        for th, wh in zip(t_hi, w_hi):
            acc += wh * float(np.dot(w_lo, _gather(u, t_lo | th)))
        out[r] = acc
    return out


# ---- formula inputs: exact integer formulas evaluated where they are gathered (torch on the device, numpy here) ----
_GOLD32 = 0x9E3779B1


def hash32(t):
    """(t * 0x9E3779B1) mod 2^32 for int64 indices t < 2^31 (exact: the product stays below 2^63)."""
    return (t * _GOLD32) & 0xFFFFFFFF


def u_hash(t):
    """u(t) = hash32(t) 2^-32 - 0.5: fp64-exact values in [-0.5, 0.5) (numpy int64 array or torch int64 tensor)."""
    h = hash32(t)
    return (h.astype(np.float64) if isinstance(h, np.ndarray) else h.double()) * 2.0 ** -32 - 0.5


def w_ties(t):
    """hash mod 4: values 0..3 with many exact ties."""
    h = hash32(t) % 4
    return h.astype(np.float64) if isinstance(h, np.ndarray) else h.double()


def w_rounding(t):
    """1e16 + 2 (hash mod 3): r_action k of order 1 is lost in the rounding of fl(r_action k) + w."""
    h = hash32(t) % 3
    return 1e16 + 2.0 * (h.astype(np.float64) if isinstance(h, np.ndarray) else h.double())


# ---- the perturbation channel over all states, for N <= 24 ----------------------------------------------------------
def kp_tensor(u, p):
    """(K_p u) over all 2^N states as a tensor product: one 2x2 contraction [[1-p, p], [p, 1-p]] per gene axis."""
    v = np.array(u, dtype=np.float64)
    n = v.size.bit_length() - 1
    q = 1.0 - p
    for i in range(n):
        x = v.reshape(-1, 2, 1 << i)
        a, z = x[:, 0, :].copy(), x[:, 1, :].copy()
        x[:, 0, :] = q * a + p * z
        x[:, 1, :] = q * z + p * a
    return v


def kp_direct(u, states, p):
    """(K_p u)(x) = sum over every perturbation mask m of p^|m| (1-p)^(N-|m|) u[x ^ m], at the listed states."""
    u = np.asarray(u, dtype=np.float64)
    n = u.size.bit_length() - 1
    m = np.arange(1 << n, dtype=np.int64)
    pc = np.zeros(m.size, dtype=np.int64)
    for i in range(n):
        pc += (m >> i) & 1
    pm = (p ** pc) * ((1.0 - p) ** (n - pc))
    return np.array([float(np.dot(pm, u[int(x) ^ m])) for x in states])


def masks_of(flip_genes, max_flips):
    genes = [g for g in range(64) if (flip_genes >> g) & 1]
    out = []
    for k in range(0, min(max_flips, len(genes)) + 1):
        for c in itertools.combinations(genes, k):
            out.append(sum(1 << g for g in c))
    return out


def improve_brute(w, flip_genes, max_flips, r_action):
    """v[s] = max_m fl(r_action |m|) + w[s ^ m] over every allowed mask; policy[s] = the first maximiser in the order
    (fewer flips, larger w[s ^ m], smaller s ^ m)."""
    w = np.asarray(w, dtype=np.float64)
    S = w.size
    s = np.arange(S, dtype=np.int64)
    best_v = np.full(S, -np.inf)
    best_k = np.zeros(S, dtype=np.int64)
    best_w = np.full(S, -np.inf)
    best_e = np.zeros(S, dtype=np.int64)
    for m in masks_of(flip_genes, max_flips):
        k = bin(m).count("1")
        e = s ^ m
        we = w[e]
        val = np.float64(r_action) * np.float64(k) + we
        better = (val > best_v) | ((val == best_v) & ((k < best_k) | ((k == best_k) & ((we > best_w) |
                                                                                        ((we == best_w) & (e < best_e))))))
        best_v = np.where(better, val, best_v)
        best_k = np.where(better, k, best_k)
        best_w = np.where(better, we, best_w)
        best_e = np.where(better, e, best_e)
    return best_v, (best_e ^ s).astype(np.int64)


def improve_brute_states(w, states, flip_genes, max_flips, r_action):
    """improve_brute evaluated only at the listed states: each state's allowed masks enumerated, ``w`` an array over
    all states or a callable on int64 indices.  Returns (v, policy) at those states."""
    s = np.asarray(states, dtype=np.int64)
    masks = np.asarray(masks_of(flip_genes, max_flips), dtype=np.int64)
    ends = s[:, None] ^ masks[None, :]
    wall = _gather(w, ends.ravel()).reshape(ends.shape)
    best_v = np.full(s.size, -np.inf)
    best_k = np.zeros(s.size, dtype=np.int64)
    best_w = np.full(s.size, -np.inf)
    best_e = np.zeros(s.size, dtype=np.int64)
    for j, m in enumerate(masks):
        k = bin(int(m)).count("1")
        e, we = ends[:, j], wall[:, j]
        val = np.float64(r_action) * np.float64(k) + we
        better = (val > best_v) | ((val == best_v) & ((k < best_k) | ((k == best_k) & ((we > best_w) |
                                                                                        ((we == best_w) & (e < best_e))))))
        best_v = np.where(better, val, best_v)
        best_k = np.where(better, k, best_k)
        best_w = np.where(better, we, best_w)
        best_e = np.where(better, e, best_e)
    return best_v, best_e ^ s


def improve_ball(w, flip_genes, max_flips, r_action):
    """The device's rule restated: B_0 = (w[s], s), B_k = best of B_{k-1} over s and its one-flip neighbours (larger
    value, then smaller endpoint); the candidate fl(r_action k) + B_k replaces the incumbent only when strictly larger."""
    w = np.asarray(w, dtype=np.float64)
    S = w.size
    s = np.arange(S, dtype=np.int64)
    bv, be = w.copy(), s.copy()
    v = np.float64(r_action) * np.float64(0) + w
    pol = np.zeros(S, dtype=np.int64)
    genes = [g for g in range(64) if (flip_genes >> g) & 1]
    for k in range(1, max_flips + 1):
        nv, ne = bv.copy(), be.copy()
        for g in genes:
            cv, ce = bv[s ^ (1 << g)], be[s ^ (1 << g)]
            better = (cv > nv) | ((cv == nv) & (ce < ne))
            nv, ne = np.where(better, cv, nv), np.where(better, ce, ne)
        bv, be = nv, ne
        cand = np.float64(r_action) * np.float64(k) + bv
        up = cand > v
        v = np.where(up, cand, v)
        pol = np.where(up, s ^ be, pol)
    return v, pol


def classify(onet_n, attractors, target):
    """(hit, wrong) over all states: in the target attractor; in another attractor and not in the target."""
    return classify_states(onet_n, attractors, target, np.arange(1 << onet_n))


def classify_states(onet_n, attractors, target, states):
    """classify restricted to the listed states."""
    offs, care, val = O.attractor_tables(attractors, onet_n)
    s = np.asarray(states, dtype=np.int64).astype(np.uint64)
    inside = []
    for a in range(len(offs) - 1):
        h = np.zeros(s.size, dtype=bool)
        for e in range(offs[a], offs[a + 1]):
            h |= (s & care[e, 0]) == val[e, 0]
        inside.append(h)
    hit = inside[target]
    other = np.zeros(s.size, dtype=bool)
    for a, h in enumerate(inside):
        if a != target:
            other |= h
    return hit, other & ~hit


def solve(P, hit, wrong, stages, flip_genes, max_flips, objective="steps", r_success=0.0, r_step=-1.0, r_action=0.0,
          r_wrong=0.0, gamma=1.0):
    """Finite-horizon backward induction with brute-force maximisation: (values [stages+1, S], policies [stages, S])."""
    if objective == "steps":
        r_success, r_step, r_action, r_wrong, gamma = 0.0, -1.0, 0.0, 0.0, 1.0
        v = np.where(hit, 0.0, -1.0)
    else:
        v = np.zeros(hit.size)
    values, policies = [v], []
    for _ in range(stages):
        u = np.where(hit, r_success, np.where(wrong, r_wrong, 0.0)) + np.where(hit, 0.0, gamma * v)
        w = P @ u
        best, pol = improve_brute(w, flip_genes, max_flips, r_action)
        v = r_step + best
        if objective == "steps":
            v = np.where(hit, 0.0, v)
        values.append(v)
        policies.append(pol)
    return np.array(values), np.array(policies)

