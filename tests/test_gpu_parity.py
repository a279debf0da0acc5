"""GPU parity: the CUDA path (through the C-ABI, via VecPBNEnv) against the CPU oracle.

Bar: bit-exact for states, counters, flags and rewards (rewards are fp32 computed with the
same two rounded operations on both sides).
"""
import hashlib
import zlib

import numpy as np
import pytest

from helpers import NETS, attractor_set, golden, k4_inputs, k4_selections, oracle_net, product_net, random_case

pytestmark = pytest.mark.gpu

KW = dict(horizon=20, r_success=5.0, r_step=-0.25, r_action=-1.0)
KERNELS = ["scalar", "sliced"]
MODES = {"none": 0, "A": 1, "B": 2, "C": 3}


def _env(name, e, mode="A", p=0.0, kernel="auto", **extra):
    from pbn_rl_b200 import VecPBNEnv
    kw = dict(KW)
    kw.update(extra)
    return VecPBNEnv(product_net(name), e, attractor_set(name), device="cuda:0", perturb_p=p, perturb_mode=mode,
                     seed=0x5EED, kernel=kernel, **kw)


def _oracle_step(name, case, sel, pert, mode, horizon=20):
    from oracle import pbn_oracle as O
    onet = oracle_net(name)
    tables = O.attractor_tables(attractor_set(name).attractors, onet.n)
    kw = dict(KW)
    kw["horizon"] = horizon
    return O.batched_step(onet, tables, case["state"], case["actions"], case["target"], case["t"],
                          mode=MODES[mode], sel=sel, pert=pert, **kw)


def _load(env, case):
    import torch
    env.set_state(torch.from_numpy(case["state"].astype(np.int64)), packed=True)
    env.set_target(torch.from_numpy(case["target"]))
    env.t.copy_(torch.from_numpy(case["t"].astype(np.int16)))


def _compare(env, expect, tag):
    import torch
    torch.cuda.synchronize()
    nxt, t1, rew, term, trunc = expect
    assert np.array_equal(env.state.cpu().numpy().astype(np.uint64), nxt), tag + ": state"
    assert np.array_equal(env.t.cpu().numpy().astype(np.uint16), t1), tag + ": t"
    assert np.array_equal(env.reward.cpu().numpy().view(np.uint32), rew.view(np.uint32)), tag + ": reward"
    assert np.array_equal(env.terminated.cpu().numpy(), term), tag + ": terminated"
    assert np.array_equal(env.truncated.cpu().numpy(), trunc), tag + ": truncated"


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("name", NETS)
def test_k4_known_answer_on_gpu(name, kernel):
    """Fixture K4 (SURVEY.md 8c): 4 x 4096 next states per network, sha256 over LE u64 words."""
    import torch
    net = product_net(name)
    n = net.n_genes
    x = k4_inputs(n)
    h = hashlib.sha256()
    from pbn_rl_b200 import VecPBNEnv
    env = VecPBNEnv(net, 4096, None, device="cuda:0", perturb_mode="none", horizon=0, kernel=kernel)
    assert env.kernel == kernel
    for sel in k4_selections(n):
        env.set_state(torch.from_numpy(x.astype(np.int64)), packed=True)
        env.step_injected(None, torch.from_numpy(sel))
        torch.cuda.synchronize()
        h.update(env.state.cpu().numpy().astype("<u8").tobytes())
    assert h.hexdigest() == golden("k4_transitions.json")[name]["sha256"]
    assert env.launches >= 4


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("name", NETS)
@pytest.mark.parametrize("mode", ["none", "A", "B", "C"])
def test_injected_step_bit_exact(name, mode, kernel):
    import torch
    e = 4096
    case = random_case(name, e, seed=zlib.crc32((name + mode).encode()) & 0xFFFF)
    env = _env(name, e, mode=mode, kernel=kernel)
    _load(env, case)
    env.step_injected(torch.from_numpy(case["actions"]), torch.from_numpy(case["sel"]),
                      torch.from_numpy(case["pert"].astype(np.int64)))
    _compare(env, _oracle_step(name, case, case["sel"], case["pert"], mode), f"{name}/{mode}/{kernel}")


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("e", [1, 31, 33, 1025, 3000])
def test_ragged_sizes(e, kernel):
    import torch
    name = "pbn28"
    case = random_case(name, e, seed=e)
    env = _env(name, e, mode="A", kernel=kernel)
    _load(env, case)
    env.step_injected(torch.from_numpy(case["actions"]), torch.from_numpy(case["sel"]),
                      torch.from_numpy(case["pert"].astype(np.int64)))
    _compare(env, _oracle_step(name, case, case["sel"], case["pert"], "A"), f"E={e}")
    # own-RNG mode on the same ragged batch
    from oracle import pbn_oracle as O
    env2 = _env(name, e, mode="A", p=0.02, kernel=kernel)
    _load(env2, case)
    env2.step(torch.from_numpy(case["actions"]).cuda())
    ids = np.arange(e, dtype=np.uint64)
    onet = oracle_net(name)
    if kernel == "scalar":
        sel, pert = O.scalar_stream_selection(onet, ids, 0, 0x5EED), O.scalar_stream_perturbation(onet.n, 0.02, ids, 0, 0x5EED)
    else:
        sel, pert = O.sliced_stream(onet, 0.02, ids, 0, 0x5EED)
    _compare(env2, _oracle_step(name, case, sel, pert, "A"), f"E={e}/philox")


def test_empty_batch_is_a_noop():
    env = _env("pbn7", 0)
    env.step(None)
    assert env.launches == 0


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("name", NETS)
@pytest.mark.parametrize("mode", ["A", "B", "C"])
def test_philox_step_bit_exact(name, mode, kernel):
    """Own-RNG mode: the oracle re-derives predictor choices and perturbation masks from the
    documented Philox streams and must land on the very same states."""
    import torch
    from oracle import pbn_oracle as O
    e, p = 4096, 0.02
    case = random_case(name, e, seed=7)
    env = _env(name, e, mode=mode, p=p, kernel=kernel)
    assert env.kernel == kernel
    onet = oracle_net(name)
    ids = np.arange(e, dtype=np.uint64)
    state = case["state"]
    t = case["t"]
    _load(env, case)
    for step in range(3):
        env.step(torch.from_numpy(case["actions"]).cuda())
        if env.kernel == "scalar":
            sel = O.scalar_stream_selection(onet, ids, step, 0x5EED)
            pert = O.scalar_stream_perturbation(onet.n, p, ids, step, 0x5EED)
        else:
            sel, pert = O.sliced_stream(onet, p, ids, step, 0x5EED)
        cur = dict(case, state=state, t=t)
        expect = _oracle_step(name, cur, sel, pert, mode)
        _compare(env, expect, f"{name}/{mode}/step{step}")
        state, t = expect[0], expect[1]
    assert pert.any(), "perturbation stream never fired: test is vacuous"


@pytest.mark.parametrize("kernel", KERNELS)
def test_sharding_invariance(kernel):
    """Two shards with env_offset 0 / 2048 reproduce the single 4096-env batch (global env ids
    drive the Philox counters)."""
    import torch
    name, e = "pbn28", 4096
    case = random_case(name, e, seed=11)
    full = _env(name, e, mode="A", p=0.01, kernel=kernel)
    _load(full, case)
    full.step(torch.from_numpy(case["actions"]).cuda())
    ref = full.state.cpu().numpy()
    for lo in (0, 2048):
        sub = {k: v[lo:lo + 2048] for k, v in case.items()}
        shard = _env(name, 2048, mode="A", p=0.01, env_offset=lo, kernel=kernel)
        _load(shard, sub)
        shard.step(torch.from_numpy(sub["actions"]).cuda())
        assert np.array_equal(shard.state.cpu().numpy(), ref[lo:lo + 2048])


@pytest.mark.parametrize("name", ["pbn7", "pbn10", "pbn28", "pbn70"])
def test_reset_matches_oracle(name):
    import torch
    from oracle import pbn_oracle as O
    e = 2048
    attrs = attractor_set(name)
    env = _env(name, e)
    state, tgt = env.reset()
    torch.cuda.synchronize()
    tables = O.attractor_tables(attrs.attractors, attrs.n_genes)
    val, src, tg = O.stream_reset(tables, len(attrs), np.arange(e, dtype=np.uint64), 0, 0x5EED)
    assert np.array_equal(state.cpu().numpy().astype(np.uint64), val)
    assert np.array_equal(tgt.cpu().numpy(), tg)
    assert np.array_equal(env.source_id.cpu().numpy(), src)
    assert (src != tg).all() and set(src.tolist()) == set(range(len(attrs)))
    ids = env.attractor_ids().cpu().numpy()
    assert np.array_equal(ids, src)  # every start state lies in its source attractor
    assert (env.t.cpu().numpy() == 0).all()


@pytest.mark.parametrize("kernel", KERNELS)
def test_autoreset_equals_step_then_reset(kernel):
    import torch
    name, e = "pbn10", 4096
    case = random_case(name, e, seed=3)
    case["t"][:] = 18
    a = _env(name, e, mode="A", p=0.01, auto_reset=True, kernel=kernel)
    b = _env(name, e, mode="A", p=0.01, auto_reset=False, kernel=kernel)
    for env in (a, b):
        _load(env, case)
    final = torch.zeros_like(a.state)
    for step in range(3):
        acts = torch.from_numpy(case["actions"]).cuda()
        a.step(acts, final_state=final)
        b.step(acts)
        assert torch.equal(final, b.state)
        done = (b.terminated | b.truncated)
        assert int(done.sum()) > 0
        b.step_ctr -= 1
        b.reset(mask=done)  # same step counter as the fused path used
        assert torch.equal(a.state, b.state) and torch.equal(a.target_id, b.target_id)
        assert torch.equal(a.t, b.t) and torch.equal(a.reward, b.reward)
    st = a.stats()
    assert st["steps"] == 3 * e and st["episodes"] == st["terminated"] + st["truncated"] > 0


def test_pack_unpack_roundtrip():
    import torch
    for name in ("pbn28", "pbn70"):
        net = product_net(name)
        e = 1000
        bits = (torch.rand(e, net.n_genes) < 0.5).to(torch.uint8)
        env = _env(name, e)
        env.set_state(bits, packed=False)
        assert torch.equal(env.unpack().cpu(), bits)
        assert torch.equal(env.unpack(dtype=torch.float32).cpu(), bits.float())
        from pbn_rl_b200 import pack_states
        assert np.array_equal(env.state.cpu().numpy().astype(np.uint64), pack_states(bits.numpy()))


def test_attractor_membership_with_wildcards():
    """data/attractors_Bittner-7.pkl stores its 4-state attractor as one tuple with two '*'."""
    import torch
    attrs = attractor_set("pbn7")
    env = _env("pbn7", 128)
    allstates = torch.arange(128, dtype=torch.int64).reshape(128, 1)
    ids = env.attractor_ids(allstates).cpu().numpy()
    expect = np.array([attrs.attractor_of([(s >> i) & 1 for i in range(7)]) for s in range(128)])
    assert np.array_equal(ids, expect)
    assert (ids >= 0).sum() == 7  # 3 singletons + 4 wildcard states (fixture K2)


@pytest.mark.parametrize("kernel", KERNELS)
def test_large_batch_properties(kernel):
    """BASELINE size (2^20 envs, Bittner-28): size-independent properties instead of a full oracle pass."""
    import torch
    name, e = "pbn28", 1 << 20
    net = product_net(name)
    env = _env(name, e, mode="A", p=0.001, auto_reset=False, kernel=kernel)
    g = torch.Generator(device="cuda").manual_seed(0)
    s0 = torch.randint(0, 1 << 28, (e, 1), generator=g, device="cuda", dtype=torch.int64)
    env.set_state(s0, packed=True)
    env.set_target(torch.randint(0, 14, (e,), generator=g, device="cuda", dtype=torch.int32))
    acts = torch.randint(0, 29, (e, 3), generator=g, device="cuda", dtype=torch.uint8)
    env.step(acts)
    s1 = env.state.clone()
    # (1) determinism: same counters, same inputs -> same outputs
    env.step_ctr = 0
    env.set_state(s0, packed=True)
    env.t.zero_()
    env.step(acts)
    assert torch.equal(env.state, s1)
    # (2) states stay inside N bits; reward takes only the values the formula allows
    assert int((s1 >> 28).abs().sum()) == 0
    vals = set(env.reward.unique().cpu().tolist())
    allowed = {KW["r_step"] + KW["r_action"] * k + h for k in range(4) for h in (0.0, KW["r_success"])}
    assert vals <= allowed
    # (3) a random 4096-env slice agrees with the oracle on the same stream
    from oracle import pbn_oracle as O
    lo = 512 * 1024
    ids = np.arange(lo, lo + 4096, dtype=np.uint64)
    onet = oracle_net(name)
    if env.kernel == "scalar":
        sel = O.scalar_stream_selection(onet, ids, 0, 0x5EED)
        pert = O.scalar_stream_perturbation(28, 0.001, ids, 0, 0x5EED)
    else:
        sel, pert = O.sliced_stream(onet, 0.001, ids, 0, 0x5EED)
    case = dict(state=s0[lo:lo + 4096].cpu().numpy().astype(np.uint64), actions=acts[lo:lo + 4096].cpu().numpy(),
                target=env.target_id[lo:lo + 4096].cpu().numpy(), t=np.zeros(4096, np.uint16))
    nxt = _oracle_step(name, case, sel, pert, "A")[0]
    assert np.array_equal(s1[lo:lo + 4096].cpu().numpy().astype(np.uint64), nxt)
    # (4) terminated envs really sit in their target attractor
    term = env.terminated.bool()
    ids_gpu = env.attractor_ids()
    assert torch.equal(ids_gpu[term], env.target_id[term])


@pytest.mark.parametrize("name,e,p", [("pbn28", 1 << 17, 1e-5), ("pbn28", 8192, 0.3), ("pbn70", 1 << 15, 2e-5),
                                      ("pbn70", 4096, 0.2), ("pbn7", 1 << 16, 3e-4), ("pbn70", 4096, 0.6)])
def test_perturbation_stream_extremes(name, e, p):
    """The geometric skip of the sliced kernel (float first guess + exact table window, binary search as
    fallback; events pre-drawn into packed words, overflow redone in phase D) against the oracle's plain walk
    over the survival table: very rare events (the float guess is least accurate) and very frequent ones
    (every thread overflows its pre-drawn list; at pbn70 and p = 0.6 a sub-stream's walk draws about 336 words, past its
    first 64 Philox blocks into the range pert_block continues it in)."""
    import torch
    from oracle import pbn_oracle as O
    case = random_case(name, e, seed=13)
    env = _env(name, e, mode="B", p=p, kernel="sliced")
    onet = oracle_net(name)
    ids = np.arange(e, dtype=np.uint64)
    state, t = case["state"], case["t"]
    _load(env, case)
    total = 0
    for step in range(2):
        env.step(torch.from_numpy(case["actions"]).cuda())
        sel, pert = O.sliced_stream(onet, p, ids, step, 0x5EED)
        expect = _oracle_step(name, dict(case, state=state, t=t), sel, pert, "B")
        _compare(env, expect, f"{name}/p={p}/step{step}")
        state, t = expect[0], expect[1]
        total += int(sum(bin(int(x)).count("1") for x in pert.reshape(-1)))
    assert total > 0, "no perturbation event in the sample: test is vacuous"
    assert env.stats()["perturbed"] == total


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("name", ["pbn10", "pbn7", "pbn28"])
def test_wrong_attractor_reward_term(name, kernel):
    """r_wrong (upstream's "-2 wrong attractor", SURVEY.md 8c): envs that end a step in an attractor other than their
    target get r_wrong instead of r_success -- rewards bit-exact against the oracle, both kernels."""
    import torch
    e = 4096
    case = random_case(name, e, seed=77)
    attrs = attractor_set(name)
    # start a third of the envs inside attractors so that hits and wrong-attractor endings both occur
    rng = np.random.default_rng(1)
    flat = [s for a in attrs.attractors for s in a]
    for k in range(0, e, 3):
        s = flat[int(rng.integers(0, len(flat)))]
        case["state"][k, :] = 0
        for i, b in enumerate(s):
            if b != "*" and int(b):
                case["state"][k, i >> 6] |= np.uint64(1) << np.uint64(i & 63)
    case["actions"][::2] = 0
    env = _env(name, e, mode="none", kernel=kernel, r_wrong=-2.0)
    _load(env, case)
    env.step_injected(torch.from_numpy(case["actions"]), torch.from_numpy(case["sel"]))
    from oracle import pbn_oracle as O
    onet = oracle_net(name)
    tables = O.attractor_tables(attrs.attractors, onet.n)
    exp = O.batched_step(onet, tables, case["state"], case["actions"], case["target"], case["t"], mode=0, sel=case["sel"],
                         pert=np.zeros_like(case["pert"]), r_wrong=-2.0, **KW)
    plain = O.batched_step(onet, tables, case["state"], case["actions"], case["target"], case["t"], mode=0, sel=case["sel"],
                           pert=np.zeros_like(case["pert"]), **KW)
    assert (exp[2] != plain[2]).sum() > 10          # the term fires
    _compare(env, exp, f"{name}/{kernel}/r_wrong")
