"""The oracle against the golden fixtures derived from the reference tree (SURVEY.md 8c K2/K4/K5)."""
import hashlib
import itertools

import numpy as np
import pytest

from helpers import NETS, attractor_set, golden, k4_inputs, k4_selections, oracle_net, product_net, random_case
from oracle import pbn_oracle as O
from oracle.philox_ref import philox_scalar


def test_philox_known_answers():
    # Random123 kat_vectors, philox4x32 10 rounds
    kat = [((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
            "d16cfe09 94fdcceb 5001e420 24126ea1")]
    for ctr, key, want in kat:
        assert " ".join("%08x" % v for v in philox_scalar(ctr, key)) == want


@pytest.mark.parametrize("name", NETS)
def test_k4_batch_transition(name):
    onet = oracle_net(name)
    x = k4_inputs(onet.n)
    zeros = np.zeros_like(x)
    h = hashlib.sha256()
    for sel in k4_selections(onet.n):
        h.update(onet.transition_batch(x, zeros, sel, zeros, O.PERT_NONE).astype("<u8").tobytes())
    assert h.hexdigest() == golden("k4_transitions.json")[name]["sha256"]


@pytest.mark.parametrize("name", NETS)
def test_k4_spot_rows_per_instance(name):
    onet = oracle_net(name)
    spot = golden("k4_transitions.json")[name]["spot_j0"]
    for mode, (s_hex, t_hex) in spot.items():
        sel = [int(mode[1])] * onet.n if mode != "mix" else [i % 3 for i in range(onet.n)]
        assert onet.transition(int(s_hex, 16), 0, sel, 0, O.PERT_NONE) == int(t_hex, 16)


def test_k2_bittner7_attractors_are_the_sink_sccs():
    """data/attractors_Bittner-7.pkl == sink SCCs of the perturbation-free STG of pbn7 (K2/K5)."""
    onet = oracle_net("pbn7")
    n = 7
    succ = {}
    for s in range(1 << n):
        nxt = set()
        for sel in itertools.product(range(3), repeat=n):
            nxt.add(onet.transition(s, 0, sel, 0, O.PERT_NONE))
        succ[s] = nxt
    # sink SCC test without a graph library: a set C is a sink SCC iff closed and strongly connected
    sinks = golden("k5_stg.json")["pbn7"]["sink_sccs"]
    for comp in sinks:
        comp = set(comp)
        for s in comp:
            assert succ[s] <= comp
        for a in comp:  # reachability inside comp
            seen, todo = {a}, [a]
            while todo:
                for t in succ[todo.pop()]:
                    if t not in seen:
                        seen.add(t)
                        todo.append(t)
            assert seen == comp
    # and the pickle's attractors expand to exactly those state sets
    attrs = golden("attractors_bittner7.json")["attractors"]
    expanded = []
    for attr in attrs:
        states = set()
        for pat in attr:
            stars = [i for i, b in enumerate(pat) if b == "*"]
            for fill in itertools.product((0, 1), repeat=len(stars)):
                bits = [0 if b == "*" else int(b) for b in pat]
                for i, v in zip(stars, fill):
                    bits[i] = v
                states.add(O.bits_to_int(bits))
        expanded.append(sorted(states))
    assert sorted(expanded) == sorted(sinks)


@pytest.mark.parametrize("name", ["pbn7", "pbn28", "pbn70"])
@pytest.mark.parametrize("mode", ["none", "A", "B", "C"])
def test_batch_matches_per_instance(name, mode):
    onet = oracle_net(name)
    case = random_case(name, 64, seed=5)
    flips = np.zeros_like(case["state"])
    out = onet.transition_batch(case["state"], flips, case["sel"], case["pert"], mode)
    for e in range(64):
        s = int(case["state"][e, 0]) | (int(case["state"][e, 1]) << 64 if onet.words == 2 else 0)
        p = int(case["pert"][e, 0]) | (int(case["pert"][e, 1]) << 64 if onet.words == 2 else 0)
        t = onet.transition(s, 0, [int(v) for v in case["sel"][e]], p, mode)
        got = int(out[e, 0]) | (int(out[e, 1]) << 64 if onet.words == 2 else 0)
        assert got == t


def test_product_lut_compiler_agrees_with_oracle_eval():
    """Two independent evaluators (truth tables vs python eval) on random states."""
    rng = np.random.default_rng(0)
    for name in NETS:
        net, onet = product_net(name), oracle_net(name)
        for _ in range(50):
            s = int(rng.integers(0, 2**62)) | (int(rng.integers(0, 2**62)) << 62)
            s &= (1 << net.n_genes) - 1
            sel = [int(rng.integers(0, len(fs))) for fs in net.functions]
            assert net.next_state_int(s, sel) == onet.transition(s, 0, sel, 0, O.PERT_NONE)


def test_batched_step_rewards_and_flags():
    name = "pbn10"
    onet = oracle_net(name)
    attrs = attractor_set(name)
    tables = O.attractor_tables(attrs.attractors, onet.n)
    case = random_case(name, 512, seed=9)
    nxt, t1, rew, term, trunc = O.batched_step(onet, tables, case["state"], case["actions"], case["target"], case["t"],
                                               horizon=20, mode=O.PERT_A, sel=case["sel"], pert=case["pert"],
                                               r_success=5.0, r_step=0.0, r_action=-1.0)
    for e in range(512):
        flip = O.flip_mask_from_actions(case["actions"][e], onet.n)
        want = onet.transition(int(case["state"][e, 0]), flip, case["sel"][e], int(case["pert"][e, 0]), O.PERT_A)
        assert int(nxt[e, 0]) == want
        hit = attrs.contains(int(case["target"][e]), O.int_to_bits(want, onet.n))
        assert bool(term[e]) == hit
        assert bool(trunc[e]) == ((not hit) and int(case["t"][e]) + 1 >= 20)
        assert rew[e] == O.reward_f32(bin(flip).count("1"), hit, 5.0, 0.0, -1.0)


def test_stream_statistics():
    """The Philox-driven selection is uniform over 3 predictors and perturbation hits at rate p."""
    onet = oracle_net("pbn28")
    ids = np.arange(20000, dtype=np.uint64)
    sel = O.scalar_stream_selection(onet, ids, 5, 0x5EED)
    for i in range(onet.n):
        counts = np.bincount(sel[:, i], minlength=3)
        chi2 = ((counts - 20000 / 3) ** 2 / (20000 / 3)).sum()
        assert chi2 < 30, (i, counts)
    p = 0.01
    pert = O.scalar_stream_perturbation(28, p, ids, 5, 0x5EED)
    nbits = sum(bin(int(x)).count("1") for x in pert[:, 0])
    mean = 20000 * 28 * p
    assert abs(nbits - mean) < 5 * np.sqrt(mean)
    assert int(pert.max()) < (1 << 28)


def test_per_instance_env_protocol():
    onet = oracle_net("pbn7")
    attrs = attractor_set("pbn7")
    env = O.OraclePBNEnv(onet, attrs.attractors, horizon=20, perturb_p=0.0, seed=1)
    (state, target), info = env.reset()
    assert len(state) == 7 and len(target) == 7 and env.is_attracting_state(state)
    assert env.state_attractor_id != env.target_attractor_id
    total = 0
    for _ in range(200):
        state, reward, term, trunc, _ = env.step([0, 3, 3])
        total += 1
        if term or trunc:
            assert term == env.in_target(state)
            (state, target), _ = env.reset()
    env.setTarget(attrs.attractors[0])
    env.set_state([1, 0, 1, 0, 0, 1, 1])
    assert env.in_target(env.render())  # wildcard positions 4,5
    s2, r, term, trunc, _ = env.step([])  # uncontrolled step inside the wildcard attractor stays inside
    assert term and r == 5.0


@pytest.mark.parametrize("name", ["pbn28", "pbn70"])
@pytest.mark.parametrize("bins", [1, 3, 8])
def test_batched_step_ignores_action_bytes_above_n(name, bins):
    """The batched flip mask equals the per-instance one for action bytes 0..255: 0 and bytes above N are no-ops,
    repeats flip once, and only the flipped genes are charged r_action."""
    onet = oracle_net(name)
    n, w, e = onet.n, onet.words, 512
    rng = np.random.default_rng(bins)
    acts = rng.integers(0, 256, size=(e, bins)).astype(np.uint8)
    acts[::4] = rng.integers(0, n + 2, size=(len(acts[::4]), bins))
    acts[1::4, 0] = n
    acts[2::4] = acts[2::4, :1]
    words = k4_inputs(n)[:e]
    sel = np.zeros((e, n), dtype=np.uint8)
    nxt, _, rew, _, _ = O.batched_step(onet, O.attractor_tables([], n), words, acts, np.full(e, -1), np.zeros(e),
                                       horizon=0, mode=0, sel=sel, pert=np.zeros((e, w), dtype=np.uint64),
                                       r_success=0.0, r_step=0.0, r_action=-1.0)
    flip = np.zeros((e, w), dtype=np.uint64)
    for i, row in enumerate(acts):
        m = O.flip_mask_from_actions(row, n)
        for wd in range(w):
            flip[i, wd] = (m >> (64 * wd)) & 0xFFFFFFFFFFFFFFFF
        assert rew[i] == -bin(m).count("1"), (i, row)
    assert np.array_equal(nxt, onet.transition_batch(words, flip, sel, np.zeros_like(flip), 0))
