"""GPU: the law every sampling path draws from, against the closed forms of tests/law_oracle.py.

The bit-exact tests pin each kernel to the oracle's Philox twin, which restates the kernel's own stream layout; a twin
written from the same wrong idea would agree bit for bit.  These tests count what the kernels produce over 2^22 envs
and compare the counts with the PBN law itself:

a. selection: probe networks (uniform K = 2, 3, 4 with many contended K = 3 pool slots; weighted K = 2..4 with
   0.999 / 0.001 and 0.3 / 0.2 / 0.5; uniform and weighted K = 5..8; K = 9..12 on the scalar kernel; probes at
   positions >= 64), every (gene, predictor) frequency and the joint law of 12 probe genes;
b. the same counts split by slice bit, and 2x2 tables of env pairs of one slice group (one perturbation sub-stream,
   and two);
c. perturbation masks of keep networks (N = 1 .. 128, p = 1e-3 .. 0.9, models A / B / C): gene x slice-bit
   frequencies, Binomial(N, p) popcounts, independence of adjacent genes and of genes 63 / 64; the negate network
   under A;
d. one-step rows of every synthetic network of tests/helpers.py plus Bittner-28 and the 70-gene network, from four
   start states, with flips, models none / A / B / C, large step counters and env offsets;
e. k-step laws (k = 1..6) of the step loop and of rollout(k) against propagate() (none / A / B) and, for model C, a
   dense matrix of the closed-form rows;
f. the reset law of reset() and of the auto-reset;
g. power: the same checks reject a probe probability 2^-7 off and p = 0.0315 tested as 0.03.

Paths, where the network is eligible: the scalar kernel, the row-format sliced kernel, the plane-resident step with 4
and 8 warps (PBN_B200_PLANES_WARPS) and rollout.  The sliced-family paths draw the same streams, so their counts are
identical and add no false alarms of their own.

Decision rule (law_oracle.Judge): every Bernoulli frequency passes when its exact two-sided binomial tail is at
least ALPHA = 1.97e-9 (the two-sided normal tail at 6 sigma), so each such check has a false-alarm probability of at
most 1.97e-9 whatever its mean -- many cells here have means of 13 to 130, where a Gaussian |z| <= 6 rule would alarm
up to 100 times more often (test_oracle_law.py::test_calibration_binomial_size computes the exact sizes).  Every
chi-square test must have p > 1e-7 (bins of expected count < 5 pooled; a count where the law says 0 fails).  The
suite makes about 2.8e5 binomial checks and 2.4e3 chi-square tests (printed per test as "LAW" lines; the identical
counts of the sliced-family paths counted again), a family-wise false-alarm probability of at most
2.8e5 * 1.97e-9 + 2.4e3 * 1e-7 = 7.9e-4 < 1e-3.  Seeds are fixed, so a pass or a fail is reproducible.

The perturbation checks found the one bias they know of: a sliced perturbation sub-stream had 64 Philox blocks, and a
dense walk (8N slots, about 8Np words) wrapped onto them once N p exceeded about 30 (|z| = 45 at gene 35 for p = 0.9
and N = 64..96).  The sub-stream now continues into blocks of its own (pert_block in csrc/philox.cuh)."""
import numpy as np
import pytest

import law_oracle as L
from helpers import CASES, make_network, oracle_net, product_net

pytestmark = pytest.mark.gpu

E = 1 << 22
SEED = 0x1A5
MODELS = [("none", 0.0), ("A", 0.03), ("B", 0.03), ("C", 0.03)]
COUNTERS = [(0, 0), (1, 1 << 40), ((1 << 32) + 5, 0), ((1 << 48) - 1, 1 << 40),
            (0, 1 << 40), (1, 0), ((1 << 32) + 5, 1 << 40), ((1 << 48) - 1, 0)]


# ---------------------------------------------------------------------------------------------- plumbing
def _nets(genes, exprs):
    from oracle import pbn_oracle as O
    from pbn_rl_b200 import PBNNetwork
    return PBNNetwork.from_expressions(genes, exprs), O.OracleNetwork(genes, exprs)


def _paths(net, rollout=True):
    """Every sampling path the network is eligible for."""
    k = max(len(f) for f in net.functions)
    out = ["scalar"]
    if net.n_genes <= 96 and k <= 8 and net.max_arity <= 12:
        out.append("sliced")
        if k <= 4:
            out += ["resident4", "resident8"]
        if rollout:
            out.append("rollout")
    return out


def _env(net, path, mode="none", p=0.0, e=E, attractors=None, monkeypatch=None, **kw):
    from pbn_rl_b200 import AttractorSet, VecPBNEnv
    n = net.n_genes
    if attractors is None:
        attractors = AttractorSet([[tuple([0] * n)]], n)
    kw.setdefault("horizon", 0)
    if path.startswith("resident"):
        monkeypatch.setenv("PBN_B200_PLANES_WARPS", path[-1])
    env = VecPBNEnv(net, e, attractors, device="cuda:0", perturb_p=p, perturb_mode=mode, seed=SEED,
                    kernel="scalar" if path == "scalar" else "sliced", resident=path.startswith("resident"), **kw)
    assert env.kernel == ("scalar" if path == "scalar" else "sliced")
    return env


def _step(env, path, actions=None):
    if path == "rollout":
        assert actions is None
        env.rollout(1, stats=False)
    else:
        env.step(actions, stats=False)


def _signed(v):
    return v - (1 << 64) if v >= 1 << 63 else v


def _words(s, w):
    return [_signed((s >> (64 * k)) & ((1 << 64) - 1)) for k in range(w)]


def _load_blocks(env, starts):
    """Envs in len(starts) contiguous blocks, block b at state starts[b]."""
    import torch
    w = env.n_words
    tab = torch.tensor([_words(s, w) for s in starts], dtype=torch.int64)
    idx = torch.arange(env.num_envs) // (env.num_envs // len(starts))
    env.set_state(tab[idx].cuda(), packed=True)


def _bits(state, genes):
    import torch
    return torch.stack([(state[:, g >> 6] >> (g & 63)) & 1 for g in genes], dim=1)


def _slice_counts(state, n, blocks, pc=None):
    """counts[block, slice bit, gene] with slice bit ((e >> 7) & 7) << 2 | (e & 3); adds each env's popcount to pc."""
    import torch
    e = state.shape[0]
    out = torch.zeros((blocks, 32, n), dtype=torch.int64, device=state.device)
    for g0 in range(0, n, 16):
        gs = list(range(g0, min(n, g0 + 16)))
        b = _bits(state, gs)
        if pc is not None:
            pc += b.sum(dim=1)
        v = b.view(blocks, e // (blocks * 1024), 8, 32, 4, len(gs)).sum(dim=(1, 3))
        out[:, :, g0:g0 + len(gs)] = v.reshape(blocks, 32, len(gs))
    return out.cpu().numpy()


def _joint(state, genes, blocks):
    """counts[block, 2^len(genes)], bin bit j = gene genes[j]."""
    import torch
    k = len(genes)
    b = _bits(state, genes)
    idx = (b << torch.arange(k, device=state.device)).sum(dim=1)
    idx += (torch.arange(state.shape[0], device=state.device) // (state.shape[0] // blocks)) << k
    return torch.bincount(idx, minlength=blocks << k).view(blocks, 1 << k).cpu().numpy()


def _pairs(state, g, blocks, stride):
    """2x2 counts [block, 4] of gene g in env pairs (e, e + stride), e with bit `stride` clear: index a + 2 b."""
    import torch
    x = _bits(state, [g])[:, 0].view(blocks, -1, 2, stride)
    idx = x[:, :, 0, :] + 2 * x[:, :, 1, :]
    idx = idx.reshape(blocks, -1) + 4 * torch.arange(blocks, device=state.device)[:, None]
    return torch.bincount(idx.reshape(-1), minlength=4 * blocks).view(blocks, 4).cpu().numpy()


def _pair_checks(judge, state, genes, law, blocks, tag):
    """law[block, gene]: env pairs inside one perturbation sub-stream (e, e ^ 1) and across two (e, e ^ 256)."""
    for stride in (1, 256):
        tables = []
        for g in genes:
            c = _pairs(state, g, blocks, stride)
            tables += [(c[b], L.product_law([law[b, g], law[b, g]])) for b in range(blocks)]
        judge.chi2(tables, "%s env pairs stride %d" % (tag, stride))


# ---------------------------------------------------------------------------------------------- a, b: selection law
W_SMALL = [[0.999, 0.001], [0.3, 0.2, 0.5], [0.1, 0.2, 0.3, 0.4], [0.001, 0.999], [0.05, 0.9, 0.05], [0.7, 0.3]]
W_WIDE = [[0.05, 0.1, 0.15, 0.3, 0.4], [0.001, 0.2, 0.2, 0.2, 0.2, 0.199], [0.3, 0.2, 0.5, 0.001, 0.1, 0.1, 0.05],
          [1, 2, 3, 4, 5, 6, 7, 8]]


def _layout(name):
    """(layout, code genes) of the probe networks."""
    u = lambda k: [1.0 / k] * k          # noqa: E731
    if name in ("k4_32", "k4_96"):
        n, code = (32, 4) if name == "k4_32" else (96, 4)
        pat = [u(3), u(2), u(3), u(4), u(3), [0.3, 0.2, 0.5], u(3), None]
        out = [None] * code
        for i in range(code, n):
            v = pat[(i - code) % 8]
            out.append(W_SMALL[((i - code) // 8) % len(W_SMALL)] if v is None else v)
        return out, code
    if name == "k8_96":
        pat = [u(5), W_WIDE[0], u(3), u(6), W_WIDE[1], u(7), W_WIDE[2], u(8), W_WIDE[3], [0.999, 0.001]]
        return [None] * 8 + [pat[i % len(pat)] for i in range(88)], 8
    if name == "k12_128":
        pat = [u(9), [0.3, 0.2, 0.5], u(10), [float(j + 1) for j in range(11)], u(12), u(2), [0.5] + [0.5 / 11] * 11,
               u(5), W_WIDE[3], [0.001] * 11 + [0.989]]
        return [None] * 12 + [pat[i % len(pat)] for i in range(116)], 12
    raise KeyError(name)


def _joint_genes(layout, code):
    """12 probe genes: four of one scalar Philox block, four K = 3 genes of sliced pool group 0, then 5..8- or
    weighted predictors, the last ones at the highest positions."""
    n = len(layout)
    probes = [i for i in range(code, n) if layout[i] is not None]
    out = [i for i in probes if (i >> 2) == (probes[4] >> 2)]
    out += [i for i in probes if len(layout[i]) == 3 and (i - code) % 4 == 0 and i not in out][:4]
    rest = [i for i in reversed(probes) if i not in out and (len(layout[i]) > 4 or len(set(layout[i])) > 1)]
    return (out + rest)[:12]


def _selection_checks(judge, state, layout, code, law, blocks, tag, slices=True, pairs=True):
    n = len(layout)
    per = E // blocks
    sc = _slice_counts(state, n, blocks)
    judge.z(sc.sum(axis=1), per, law, tag + " genes")
    if slices:
        judge.z(sc, per // 32, law[:, None, :], tag + " genes x slice bit")
    genes = _joint_genes(layout, code)
    jc = _joint(state, genes, blocks)
    judge.chi2([(jc[b], L.product_law(law[b, genes])) for b in range(blocks)], tag + " joint %s" % genes)
    if pairs:
        _pair_checks(judge, state, genes[:6], law, blocks, tag)


@pytest.mark.parametrize("name", ["k4_32", "k4_96", "k8_96", "k12_128"])
def test_selection_law(name, monkeypatch):
    import torch
    layout, code = _layout(name)
    net, _ = _nets(*L.probe_network(layout, code))
    blocks = 1 << (code - 1).bit_length()
    law = np.zeros((blocks, len(layout)))
    law[:code] = L.probe_law(layout, code)
    starts = [1 << j if j < code else 0 for j in range(blocks)]
    judge = L.Judge("selection " + name)
    ref = None
    for path in _paths(net):
        env = _env(net, path, monkeypatch=monkeypatch)
        _load_blocks(env, starts)
        env.step_ctr = 3
        _step(env, path)
        st = env.state.clone()
        env.close()
        sliced = path != "scalar"
        _selection_checks(judge, st, layout, code, law, blocks, "%s %s" % (name, path), slices=sliced, pairs=sliced)
        if path == "sliced":
            ref = st
        elif sliced:
            judge.exact(torch.equal(st, ref), "%s %s: differs from the row-format sliced step" % (name, path))
        del st
    judge.check()


# ---------------------------------------------------------------------------------------------- c: perturbation law
def _perturbation_checks(judge, state, n, p, start, tag, slices=True):
    """The mask law of one run: state ^ start is the mask (keep network)."""
    import torch
    w = state.shape[1]
    m = state ^ torch.tensor(_words(start, w), dtype=torch.int64, device=state.device)
    pc = torch.zeros(state.shape[0], dtype=torch.int64, device=state.device)
    sc = _slice_counts(m, n, 1, pc)[0]
    judge.z(sc.sum(axis=0), E, p, tag + " genes")
    if slices:
        judge.z(sc, E // 32, p, tag + " genes x slice bit")
        judge.z(sc.sum(axis=1), n * (E // 32), p, tag + " slice bits")
    judge.chi2((torch.bincount(pc, minlength=n + 1).cpu().numpy(), L.binomial_pmf(n, p)), tag + " popcount")
    if n > 1:
        both = L.product_law([p, p])
        tables = [(c, both) for c in (_joint(m, [g, g + 1], 1)[0] for g in range(n - 1))]
        judge.chi2(tables, tag + " adjacent genes")
    if n > 64:
        judge.chi2((_joint(m, [63, 64], 1)[0], L.product_law([p, p])), tag + " genes 63 / 64")
    if slices:
        law = np.full((1, n), p)
        _pair_checks(judge, m, sorted({0, n // 2, n - 1}), law, 1, tag)


@pytest.mark.parametrize("n", [1, 28, 64, 65, 96, 128])
def test_perturbation_law(n, monkeypatch):
    import torch
    net, _ = _nets(*L.keep_network(n))
    judge = L.Judge("perturbation n=%d" % n)
    start = 0
    for p in (1e-3, 0.03, 0.25, 0.9):
        for mode in ("A", "B", "C"):
            ref = None
            for path in _paths(net):
                env = _env(net, path, mode, p, monkeypatch=monkeypatch)
                _load_blocks(env, [start])
                env.step_ctr = 7
                _step(env, path)
                st = env.state.clone()
                env.close()
                tag = "keep%d %s p=%g %s" % (n, mode, p, path)
                if path in ("scalar", "sliced"):
                    _perturbation_checks(judge, st, n, p, start, tag, slices=path == "sliced")
                if path == "sliced":
                    ref = st
                elif path != "scalar":
                    judge.exact(torch.equal(st, ref), tag + ": differs from the row-format sliced step")
    judge.check()


@pytest.mark.parametrize("n", [28, 96])
def test_negate_network_model_a(n, monkeypatch):
    """All genes not x_i under A: an unperturbed step negates every gene, a perturbed one skips the update, so
    popcount(t ^ s) follows law_oracle.negate_flip_law and no env stays at s."""
    import torch
    net, _ = _nets(*L.negate_network(n))
    s = int(np.random.default_rng(n).integers(0, 1 << 62)) * 3 % (1 << n)
    judge = L.Judge("negate n=%d" % n)
    for p in (0.03, 0.25):
        for path in _paths(net):
            env = _env(net, path, "A", p, monkeypatch=monkeypatch)
            _load_blocks(env, [s])
            _step(env, path)
            st = env.state
            x = st ^ torch.tensor(_words(s, st.shape[1]), dtype=torch.int64, device=st.device)
            pc = torch.zeros(E, dtype=torch.int64, device=st.device)
            _slice_counts(x, n, 1, pc)
            counts = torch.bincount(pc, minlength=n + 1).cpu().numpy()
            judge.exact(counts[0] == 0, "negate%d p=%g %s: %d envs stayed at s" % (n, p, path, counts[0]))
            if path in ("scalar", "sliced"):
                judge.chi2((counts, L.negate_flip_law(n, p)), "negate%d p=%g %s" % (n, p, path))
            env.close()
    judge.check()


# ---------------------------------------------------------------------------------------------- d: one-step rows
ROW_NETS = [c[:5] for c in CASES] + ["pbn28", "pbn70"]


def _row_net(case):
    from oracle import pbn_oracle as O
    if isinstance(case, str):
        return product_net(case), oracle_net(case), 3
    n, kmax, amax, bins, uniform = case
    genes, exprs = make_network(n, kmax, amax, seed=1000 + n, uniform=uniform)
    return _nets(genes, exprs)[0], O.OracleNetwork(genes, exprs), bins


def _row_starts(onet, rng):
    n = onet.n
    cand = [int.from_bytes(rng.bytes(16), "little") % (1 << n) for _ in range(4096)]
    q = L.q_states(onet, cand)
    free = ((q > 0.0) & (q < 1.0)).sum(axis=1)
    return [cand[int(free.argmax())], 0, (1 << n) - 1, int.from_bytes(rng.bytes(16), "little") % (1 << n)]


def _row_checks(judge, st, onet, starts, flips, mode, p, rng, tag):
    import torch
    n, w = onet.n, st.shape[1]
    blocks = len(starts)
    per = E // blocks
    sc = _slice_counts(st, n, blocks).sum(axis=1)
    for b, (s, f) in enumerate(zip(starts, flips)):
        part = st[b * per:(b + 1) * per]
        judge.z(sc[b], per, L.marginals(onet, s, f, mode, p), "%s block %d marginals" % (tag, b))
        genes, law, fixed = L.full_row(onet, s, f, mode, p)
        if len(genes) <= 16:
            mask = ((1 << n) - 1) & ~sum(1 << g for g in genes)
            mw = torch.tensor(_words(mask, w), dtype=torch.int64, device=st.device)
            fw = torch.tensor(_words(fixed, w), dtype=torch.int64, device=st.device)
            off = int(((part & mw) != fw).any(dim=1).sum())
            judge.exact(off == 0, "%s block %d: %d envs off the fixed genes" % (tag, b, off))
            if genes:
                judge.chi2((_joint(part, genes, 1)[0], law), "%s block %d full row" % (tag, b))
        else:
            proj = (genes + [g for g in rng.permutation(n).tolist() if g not in genes])[:12]
            proj = [int(g) for g in rng.permutation(proj)]
            judge.chi2((_joint(part, proj, 1)[0], L.projection(onet, s, f, mode, p, proj)),
                       "%s block %d projection %s" % (tag, b, proj))


@pytest.mark.parametrize("case", ROW_NETS, ids=[c if isinstance(c, str) else "n%d_k%d_a%d" % c[:3] for c in ROW_NETS])
def test_one_step_rows(case, monkeypatch):
    import torch
    net, onet, bins = _row_net(case)
    n = net.n_genes
    rng = np.random.default_rng(n * 7 + bins)
    starts = _row_starts(onet, rng)
    flips, acts = [], np.zeros((4, bins), dtype=np.uint8)
    for b in range(4):
        gs = rng.choice(n, size=min(b % 3 + 1, n, bins), replace=False)
        acts[b, :len(gs)] = gs + 1
        flips.append(sum(1 << int(g) for g in gs))
    actions = torch.from_numpy(np.repeat(acts, E // 4, axis=0)).cuda()
    judge = L.Judge("rows %s" % (case if isinstance(case, str) else "n=%d" % n))
    run = 0
    for path in _paths(net):
        for mode, p in MODELS:
            ctr, offset = COUNTERS[run % len(COUNTERS)]
            run += 1
            env = _env(net, path, mode, p, bins=bins, env_offset=offset, monkeypatch=monkeypatch)
            if path == "rollout":
                _load_blocks(env, [s ^ f for s, f in zip(starts, flips)])
            else:
                _load_blocks(env, starts)
            env.step_ctr = ctr
            _step(env, path, None if path == "rollout" else actions)
            st = env.state.clone()
            env.close()
            tag = "%s %s p=%g ctr=%d offset=%d" % (path, mode, p, ctr, offset)
            _row_checks(judge, st, onet, starts, flips, mode, p, rng, tag)
    judge.check()


# ---------------------------------------------------------------------------------------------- e: k-step laws
K_NETS = {
    "k2": (12, 2, 3, True), "k3": (12, 3, 4, True), "k4w": (12, 4, 4, False), "k8w": (12, 8, 3, False),
    "wide": (12, 3, 9, False), "n20": (20, 3, 4, True), "n24": (24, 2, 3, True),
}


def _k_net(name):
    n, kmax, amax, uniform = K_NETS[name]
    return _nets(*make_network(n, kmax, amax, seed=500 + n + kmax + amax, uniform=uniform))


def _k_sampled(net, path, mode, p, s0, ks, monkeypatch):
    """State tensors after k = 1..max(ks) steps of the path from the point mass s0 (rollout(k) afresh for each k)."""
    if path == "rollout":
        env = _env(net, path, mode, p, monkeypatch=monkeypatch)
        for k in ks:
            _load_blocks(env, [s0])
            env.step_ctr = 100 * k
            env.rollout(k, stats=False)
            yield k, env.state
        env.close()
        return
    env = _env(net, path, mode, p, monkeypatch=monkeypatch)
    _load_blocks(env, [s0])
    for k in ks:
        _step(env, path)
        yield k, env.state
    env.close()


@pytest.mark.parametrize("name", list(K_NETS))
def test_k_step_laws(name, monkeypatch):
    import torch
    from pbn_rl_b200 import propagate
    net, onet = _k_net(name)
    n = net.n_genes
    rng = np.random.default_rng(n)
    s0 = int(rng.integers(0, 1 << n))
    genes = [int(g) for g in rng.permutation(n)[:10]]
    judge = L.Judge("k-step " + name)
    ks = list(range(1, 7))
    for mode, p in (("none", 0.0), ("A", 0.05), ("B", 0.05)):
        one = _env(net, "scalar", mode, p, e=1)
        dists = propagate(one, s0, 6, keep=True)
        one.close()
        for path in _paths(net):
            for k, st in _k_sampled(net, path, mode, p, s0, ks, monkeypatch):
                tag = "%s %s p=%g k=%d" % (path, mode, p, k)
                if n <= 12:
                    counts = torch.bincount(st[:, 0], minlength=1 << n).cpu().numpy()
                    judge.chi2((counts, dists[k].probs.cpu().numpy()), tag + " full distribution")
                else:
                    m = dists[k].marginals()
                    judge.z(_slice_counts(st, n, 1)[0].sum(axis=0), E, m, tag + " marginals")
                    judge.chi2((_joint(st, genes, 1)[0], dists[k].projection(genes)), tag + " projection")
        del dists
        torch.cuda.empty_cache()
    judge.check()


def test_k_step_law_model_c(monkeypatch):
    """Model C (propagate does not take it): x P^k with P built from the closed-form product rows, N = 8."""
    import torch
    net, onet = _nets(*make_network(8, 4, 3, seed=88, uniform=False))
    P = L.dense_matrix(onet, "C", 0.05)
    s0 = 0b10110010
    x = np.zeros(256)
    x[s0] = 1.0
    want = {}
    for k in range(1, 7):
        x = x @ P
        want[k] = x.copy()
    judge = L.Judge("k-step model C")
    for path in _paths(net):
        for k, st in _k_sampled(net, path, "C", 0.05, s0, range(1, 7), monkeypatch):
            judge.chi2((torch.bincount(st[:, 0], minlength=256).cpu().numpy(), want[k]), "%s C k=%d" % (path, k))
    judge.check()


# ---------------------------------------------------------------------------------------------- f: reset law
def _reset_attractors(a, n, rng):
    """a attractors of 1..3 distinct entries; about half the entries carry wildcards (read as 0 by the reset)."""
    out = []
    for _ in range(a):
        vals = rng.choice(1 << n, size=int(rng.integers(1, 4)), replace=False)
        attr = []
        for v in vals:
            bits = [int(v >> i) & 1 for i in range(n)]
            if rng.random() < 0.5:
                zeros = [i for i in range(n) if not bits[i]]
                for i in rng.choice(zeros, size=min(2, len(zeros)), replace=False):
                    bits[int(i)] = "*"
            attr.append(tuple(bits))
        out.append(attr)
    return out


def _reset_counts(env, attrs):
    """counts[source, target, entry] of the current state / source_id / target_id; -1 entries (the state is no entry of
    the source) are counted in the last return value."""
    import torch
    a = len(attrs)
    m = max(len(x) for x in attrs)
    entries = L.reset_entries(attrs)
    st, src, tgt = env.state[:, 0], env.source_id.long(), env.target_id.long()
    ent = torch.full_like(src, -1)
    for s, vals in enumerate(entries):
        for j, v in enumerate(vals):
            ent = torch.where((src == s) & (st == v), torch.full_like(ent, j), ent)
    bad = int(((ent < 0) | (src < 0) | (src >= a) | (tgt < 0) | (tgt >= a)).sum())
    idx = (src.clamp(0, a - 1) * a + tgt.clamp(0, a - 1)) * m + ent.clamp(min=0)
    return torch.bincount(idx, minlength=a * a * m).view(a, a, m).cpu().numpy(), bad


@pytest.mark.parametrize("a", [2, 3, 4, 5, 6, 7, "weighted"])
def test_reset_law(a, monkeypatch):
    import torch
    from pbn_rl_b200 import AttractorSet
    n = 10
    net, _ = _nets(*L.keep_network(n))
    rng = np.random.default_rng(7 if a == "weighted" else a)
    size = 5 if a == "weighted" else a
    attrs = _reset_attractors(size, n, rng)
    pw = None
    if a == "weighted":
        pw = rng.random((size, size)) * (rng.random((size, size)) < 0.6)
        pw[0, 0], pw[1, 2], pw[3, 3], pw[4, 0] = 0.7, 0.0, 0.2, 0.0
    law = L.reset_law(attrs, pw)
    judge = L.Judge("reset %s" % a)
    aset = AttractorSet(attrs, n)
    for path in _paths(net, rollout=False):
        for how in ("reset", "auto"):
            if how == "reset" and path.startswith("resident"):
                continue
            env = _env(net, path, "A", 0.0, attractors=aset, monkeypatch=monkeypatch, horizon=1,
                       auto_reset=how == "auto", pair_weights=pw)
            if how == "reset":
                env.step_ctr = 11
                env.reset()
            else:
                env.set_state(torch.full((E, 1), (1 << n) - 1, dtype=torch.int64), packed=True)
                env.set_target(torch.zeros(E, dtype=torch.int32))
                env.step_ctr = 12
                env.step(None, stats=False)      # horizon 1: every env finishes and is reset
                judge.exact(bool((env.t == 0).all()), "%s auto: t not reset" % path)
            counts, bad = _reset_counts(env, attrs)
            env.close()
            tag = "reset %s %s %s" % (a, path, how)
            judge.exact(bad == 0, "%s: %d envs outside the reset law's support" % (tag, bad))
            judge.chi2((counts, law), tag)
    judge.check()


# ---------------------------------------------------------------------------------------------- g: power
def test_power_selection_probe_off_by_2_7(monkeypatch):
    """An env whose ASSA-like probe gene selects 0.3 + 2^-7 / 0.2 - 2^-7 / 0.5 fails the selection checks of the law
    0.3 / 0.2 / 0.5 on the scalar and the sliced kernel (and passes its own law)."""
    layout, code = _layout("k4_32")
    off = [list(v) if v is not None else None for v in layout]
    g = next(i for i in range(code, len(layout)) if layout[i] == [0.3, 0.2, 0.5])
    off[g] = [0.3 + 2.0 ** -7, 0.2 - 2.0 ** -7, 0.5]
    net, _ = _nets(*L.probe_network(off, code))
    law = L.probe_law(layout, code)
    own = L.probe_law(off, code)
    starts = [1 << j for j in range(code)]
    for path in ("scalar", "sliced"):
        env = _env(net, path, monkeypatch=monkeypatch)
        _load_blocks(env, starts)
        _step(env, path)
        st = env.state.clone()
        env.close()
        wrong, right = L.Judge("power selection %s" % path), L.Judge("own law %s" % path)
        _selection_checks(wrong, st, layout, code, law, code, path, slices=False, pairs=False)
        _selection_checks(right, st, off, code, own, code, path, slices=False, pairs=False)
        print(wrong.report(), wrong.failures[:3])
        assert wrong.failures and any("genes" in f for f in wrong.failures), wrong.report()
        right.check()


def test_power_perturbation_rate(monkeypatch):
    """An env at p = 0.0315 fails the perturbation checks of p = 0.03 (keep network, 28 genes, both kernels)."""
    net, _ = _nets(*L.keep_network(28))
    for path in ("scalar", "sliced"):
        env = _env(net, path, "A", 0.0315, monkeypatch=monkeypatch)
        _load_blocks(env, [0])
        _step(env, path)
        st = env.state.clone()
        env.close()
        wrong, right = L.Judge("power p %s" % path), L.Judge("own p %s" % path)
        _perturbation_checks(wrong, st, 28, 0.03, 0, path, slices=False)
        _perturbation_checks(right, st, 28, 0.0315, 0, path, slices=False)
        print(wrong.report(), wrong.failures[:3])
        assert wrong.min_p < 1e-7 and wrong.max_z > 6.0, wrong.report()
        right.check()
