"""Shared fixtures for the tests: golden networks, oracle twins, seeded inputs."""
import json
from functools import lru_cache
from pathlib import Path

import numpy as np

GOLD = Path(__file__).resolve().parent / "golden"
NETS = ("pbn7", "pbn10", "pbn28", "pbn70")


@lru_cache(maxsize=None)
def product_net(name):
    from pbn_rl_b200 import PBNNetwork
    return PBNNetwork.from_json(GOLD / f"{name}.json")


@lru_cache(maxsize=None)
def oracle_net(name):
    from oracle.pbn_oracle import OracleNetwork
    return OracleNetwork.from_json(GOLD / f"{name}.json")


def golden(name):
    return json.loads((GOLD / name).read_text())


@lru_cache(maxsize=None)
def attractor_set(name):
    """Attractor table used with each golden network (SURVEY.md 8c/8d):
    pbn7 -> data/attractors_Bittner-7.pkl; pbn10 -> the 3 sink SCCs (K5);
    pbn28 -> data/attractors_Bittner-28.pkl permuted to file order (K3);
    pbn70 -> 16 synthetic single-state targets from a seeded uncontrolled oracle-free construction."""
    from pbn_rl_b200 import AttractorSet, sorted_id_permutation
    net = product_net(name)
    if name == "pbn7":
        return AttractorSet([[tuple(s) for s in a] for a in golden("attractors_bittner7.json")["attractors"]], 7)
    if name == "pbn10":
        sinks = golden("k5_stg.json")["pbn10"]["sink_sccs"]
        return AttractorSet([[tuple((s >> i) & 1 for i in range(10)) for s in m] for m in sinks], 10)
    if name == "pbn28":
        raw = AttractorSet([[tuple(s) for s in a] for a in golden("attractors_bittner28.json")["attractors"]], 28)
        return raw.permuted(sorted_id_permutation(net.genes))
    rng = np.random.default_rng(70)
    states = rng.integers(0, 2, size=(16, 70))
    return AttractorSet([[tuple(int(v) for v in s)] for s in states], 70)


def k4_inputs(n):
    mask_lo = (1 << min(n, 64)) - 1
    mask_hi = (1 << (n - 64)) - 1 if n > 64 else 0
    w = 1 if n <= 64 else 2
    out = np.zeros((4096, w), dtype=np.uint64)
    for j in range(4096):
        out[j, 0] = ((j + 1) * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF & mask_lo
        if w == 2:
            out[j, 1] = ((j + 1) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF & mask_hi
    return out


def k4_selections(n):
    """The four selection modes of fixture K4, in hash order."""
    j = np.arange(4096)[:, None]
    i = np.arange(n)[None, :]
    return [np.full((4096, n), k, dtype=np.uint8) for k in range(3)] + [((i + j) % 3).astype(np.uint8)]


def random_case(name, e, seed, pert_density=0.05, sel_max=3):
    """Seeded random inputs for one step of E envs."""
    net = product_net(name)
    n, w = net.n_genes, net.n_words
    rng = np.random.default_rng(seed)
    masks = np.array(net.state_mask(), dtype=np.uint64)
    state = rng.integers(0, 2**63, size=(e, w), dtype=np.int64).astype(np.uint64) * np.uint64(2) + \
        rng.integers(0, 2, size=(e, w)).astype(np.uint64)
    state &= masks
    actions = rng.integers(0, n + 1, size=(e, 3), dtype=np.uint8)
    sel = np.zeros((e, n), dtype=np.uint8)
    for i, fs in enumerate(net.functions):
        sel[:, i] = rng.integers(0, min(len(fs), sel_max), size=e)
    pert_bits = rng.random((e, n)) < pert_density
    pert = np.zeros((e, w), dtype=np.uint64)
    for i in range(n):
        pert[:, i >> 6] |= pert_bits[:, i].astype(np.uint64) << np.uint64(i & 63)
    keep = rng.random(e) < 0.5  # half the envs unperturbed, so PERT_A exercises both branches
    pert[keep] = 0
    n_attr = len(attractor_set(name))
    target = rng.integers(0, n_attr, size=e, dtype=np.int32)
    t = rng.integers(0, 25, size=e).astype(np.uint16)
    return dict(state=state, actions=actions, sel=sel, pert=pert, target=target, t=t)


# ---- random networks at the edges of what the ABI admits (test_gpu_synthetic.py, test_gpu_edges.py)
def _sop(names, table):
    """Sum-of-products expression string for a truth table over `names` (bit j of the row index = names[j])."""
    k = len(names)
    rows = [a for a in range(1 << k) if (table >> a) & 1]
    if k == 0 or not rows:
        return "( %s & ~ %s )" % (names[0] if names else "x0", names[0] if names else "x0") if not rows else "( x0 | ~ x0 )"
    if len(rows) == 1 << k:
        return "( %s | ~ %s )" % (names[0], names[0])
    terms = []
    for a in rows:
        terms.append("( " + " & ".join(("%s" if (a >> j) & 1 else "~ %s") % names[j] for j in range(k)) + " )")
    return " | ".join(terms)


def make_network(n, kmax, amax, seed, uniform=True):
    rng = np.random.default_rng(seed)
    genes = ["x%d" % i for i in range(n)]
    exprs = []
    for i in range(n):
        k = int(rng.integers(1, kmax + 1))
        row = []
        weights = np.ones(k) if uniform else rng.integers(1, 6, size=k).astype(float)
        for f in range(k):
            ar = int(rng.integers(0, min(amax, n) + 1))
            ins = sorted(rng.choice(n, size=ar, replace=False).tolist())
            table = int(rng.integers(0, 1 << min(1 << ar, 62))) | (int(rng.integers(0, 1 << 62)) << 62 if ar > 5 else 0)
            table &= (1 << (1 << ar)) - 1
            if ar >= 7:   # keep the expression strings of wide predictors short: few minterms
                table = 0
                for a in rng.integers(0, 1 << ar, size=5):
                    table |= 1 << int(a)
            row.append((_sop([genes[j] for j in ins], table), float(weights[f] / weights.sum())))
        exprs.append(row)
    return genes, exprs


def window_network(n, k, seed):
    """A network whose free-gene count per state is set by the state: gene i has the copy predictor x_i and
    x_i XOR (x_{i+1} & ... & x_{i+k}) (indices mod n), with seeded unequal selection probabilities.  Gene i is free
    exactly when its window of k genes is all ones; otherwise both predictors keep x_i.  So a state whose ones form one
    cyclic run of length L >= k (L < n) has L - k + 1 free genes, the all-ones state has n, and the total successor
    count sum_x 2^free(x) is the trace of the n-th power of a 2^k-state transfer matrix.  k = 6 makes 7-input
    (wide) predictors."""
    rng = np.random.default_rng(seed)
    genes = ["x%d" % i for i in range(n)]
    exprs = []
    for i in range(n):
        win = " & ".join(genes[(i + j) % n] for j in range(1, k + 1))
        xor = "( %s & ~ ( %s ) ) | ( ~ %s & ( %s ) )" % (genes[i], win, genes[i], win)
        p = float(rng.uniform(0.15, 0.85))
        while abs(p - 0.5) < 0.05:
            p = float(rng.uniform(0.15, 0.85))
        exprs.append([(genes[i], p), (xor, 1.0 - p)])
    return genes, exprs


def run_state(n, start, length):
    """The state whose ones are the cyclic run of ``length`` genes from gene ``start`` (indices mod n)."""
    s = 0
    for j in range(length):
        s |= 1 << ((start + j) % n)
    return s


def make_attractors(n, count, seed):
    rng = np.random.default_rng(seed)
    out = []
    for a in range(count):
        states = []
        for _ in range(int(rng.integers(1, 4))):
            s = [int(v) for v in rng.integers(0, 2, size=n)]
            if a % 2 and n > 2:
                for j in rng.choice(n, size=min(2, n), replace=False):
                    s[int(j)] = "*"
            states.append(tuple(s))
        out.append(states)
    return out


CASES = [
    # n, kmax, amax, bins, uniform, kernels
    (1, 3, 1, 1, True, ("sliced", "scalar")),
    (2, 4, 2, 3, True, ("sliced", "scalar")),
    (31, 3, 4, 3, True, ("sliced", "scalar")),
    (32, 4, 5, 8, True, ("sliced", "scalar")),
    (33, 2, 6, 2, True, ("sliced", "scalar")),
    (64, 3, 4, 3, True, ("sliced", "scalar")),
    (65, 3, 4, 3, True, ("sliced", "scalar")),
    (96, 2, 3, 4, True, ("sliced", "scalar")),
    (97, 3, 3, 3, True, ("scalar",)),           # more than 96 genes: general kernel only
    (128, 2, 4, 5, True, ("scalar",)),
    (20, 5, 3, 3, False, ("sliced", "scalar")),  # five predictors, real selection probabilities: third selection plane
    (26, 8, 4, 3, True, ("sliced", "scalar")),   # up to eight predictors, uniform
    (12, 9, 3, 3, True, ("scalar",)),            # more than eight predictors: general kernel only
    (24, 2, 9, 3, False, ("sliced", "scalar")),  # wide predictors (7..9 inputs), weighted selection
    (40, 3, 12, 3, True, ("sliced", "scalar")),  # up to 12 inputs, two-word states
    (20, 2, 14, 3, True, ("scalar",)),           # more than 12 inputs: general kernel only
]
