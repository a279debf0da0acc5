"""GPU: pbn_step_host (host buffers; the batch cut into lanes that each run upload / kernel / download on their own
stream) against pbn_step on the same inputs -- the result must not depend on the number of lanes, the result form, the
counter mode or the kernel."""
import numpy as np
import pytest

from helpers import attractor_set, product_net

pytestmark = pytest.mark.gpu

KW = dict(horizon=6, bins=3, perturb_p=0.01, perturb_mode="A", seed=77)


def _mk(name, e, **kw):
    from pbn_rl_b200 import VecPBNEnv
    args = dict(KW)
    args.update(kw)
    return VecPBNEnv(product_net(name), e, attractor_set(name), device="cuda:0", **args)


def _seed_env(env, name, e, seed):
    import torch
    net = product_net(name)
    rng = np.random.default_rng(seed)
    masks = np.array(net.state_mask(), dtype=np.uint64)
    st = (rng.integers(0, 2**63, size=(e, net.n_words), dtype=np.int64).astype(np.uint64) * np.uint64(2)) & masks
    env.set_state(torch.from_numpy(st.astype(np.int64)), packed=True)
    env.set_target(torch.from_numpy(rng.integers(0, len(attractor_set(name)), size=e, dtype=np.int32)))


@pytest.mark.parametrize("name,e", [("pbn28", 5000), ("pbn28", 8192), ("pbn70", 3000), ("pbn10", 1)])
@pytest.mark.parametrize("kernel", ["auto", "scalar"])
@pytest.mark.parametrize("chunks", [0, 1, 3, 16])
def test_step_host_equals_step(name, e, kernel, chunks):
    import torch
    ref = _mk(name, e, kernel=kernel, auto_reset=True)
    dut = _mk(name, e, kernel=kernel, auto_reset=True)
    _seed_env(ref, name, e, 5)
    _seed_env(dut, name, e, 5)
    rng = np.random.default_rng(9)
    n = product_net(name).n_genes
    for step in range(8):
        act = rng.integers(0, n + 1, size=(e, 3), dtype=np.uint8)
        ref.step(torch.from_numpy(act).cuda())
        if step % 2:
            pinned = dut.pinned_actions()
            pinned.numpy()[...] = act
            out = dut.step_host(pinned, chunks=chunks)   # pinned tensor: used in place
        else:
            out = dut.step_host(act, chunks=chunks)      # pageable numpy array: copied into a pinned buffer
        torch.cuda.synchronize()
        assert np.array_equal(out["state"], ref.state.cpu().numpy())
        assert np.array_equal(out["reward"], ref.reward.cpu().numpy())
        assert np.array_equal(out["terminated"], ref.terminated.cpu().numpy())
        assert np.array_equal(out["truncated"], ref.truncated.cpu().numpy())
        assert np.array_equal(dut.t.cpu().numpy(), ref.t.cpu().numpy())
        assert np.array_equal(dut.target_id.cpu().numpy(), ref.target_id.cpu().numpy())
    assert ref.stats() == dut.stats()
    ref.close()
    dut.close()


@pytest.mark.parametrize("mode", ["device_counter", "pdl"])
def test_step_host_counter_modes(mode):
    """The lanes of one logical step share one Philox step counter, whichever side keeps it."""
    import torch
    e, name = 6 * 1024 + 17, "pbn28"
    ref = _mk(name, e)                                    # host-side counter
    dut = _mk(name, e, device_counter=True, pdl=(mode == "pdl"))
    _seed_env(ref, name, e, 3)
    _seed_env(dut, name, e, 3)
    rng = np.random.default_rng(4)
    for step in range(5):
        act = rng.integers(0, 29, size=(e, 3), dtype=np.uint8)
        ref.step(torch.from_numpy(act).cuda())
        out = dut.step_host(act, chunks=4)
        assert np.array_equal(out["state"], ref.state.cpu().numpy()), step
    if mode == "device_counter":
        assert int(dut.step_ctr_dev.item()) == 5
    ref.close()
    dut.close()


def test_step_host_no_actions():
    import torch
    e, name = 2048, "pbn10"
    ref, dut = _mk(name, e), _mk(name, e)
    _seed_env(ref, name, e, 1)
    _seed_env(dut, name, e, 1)
    ref.step(None)
    out = dut.step_host(None)
    torch.cuda.synchronize()
    assert np.array_equal(out["state"], ref.state.cpu().numpy())
    ref.close()
    dut.close()


def test_step_host_pageable_buffers_use_copy_engine():
    """The C entry point also takes pageable host memory (plain numpy arrays): same results."""
    import ctypes as C
    import torch
    from pbn_rl_b200 import _cabi
    e, name = 3 * 1024 + 5, "pbn28"
    ref, dut = _mk(name, e), _mk(name, e)
    _seed_env(ref, name, e, 8)
    _seed_env(dut, name, e, 8)
    act = np.random.default_rng(2).integers(0, 29, size=(e, 3), dtype=np.uint8)
    ref.step(torch.from_numpy(act).cuda())
    out = {k: np.zeros(e, dt) for k, dt in (("state", np.int64), ("reward", np.float32), ("terminated", np.uint8),
                                            ("truncated", np.uint8))}
    d_act = torch.empty((e, 3), dtype=torch.uint8, device="cuda:0")
    io = _cabi.HostIO()
    io.actions, io.actions_dev = act.ctypes.data, d_act.data_ptr()
    io.state, io.reward = out["state"].ctypes.data, out["reward"].ctypes.data
    io.terminated, io.truncated = out["terminated"].ctypes.data, out["truncated"].ctypes.data
    io.n_chunks = 2
    a = dut._args(None, None, True)
    _cabi.check(dut.lib.pbn_step_host(dut._h, C.byref(a), C.byref(io), dut._stream()))
    assert np.array_equal(out["state"], ref.state.cpu().numpy()[:, 0])
    assert np.array_equal(out["reward"], ref.reward.cpu().numpy())
    assert np.array_equal(out["terminated"], ref.terminated.cpu().numpy())
    # compact outputs are refused for pageable memory, loudly
    done = np.zeros(e, np.uint8)
    io.done = done.ctypes.data
    with pytest.raises(_cabi.PbnError):
        _cabi.check(dut.lib.pbn_step_host(dut._h, C.byref(a), C.byref(io), dut._stream()))
    ref.close()
    dut.close()


@pytest.mark.parametrize("e", [1, 1023, 4099, 65536 + 3])
def test_step_host_compact_results(e):
    """compact=True: uint32 state + reward + done byte carry the same information."""
    import torch
    name = "pbn28"
    ref, dut = _mk(name, e, auto_reset=True), _mk(name, e, auto_reset=True)
    _seed_env(ref, name, e, 11)
    _seed_env(dut, name, e, 11)
    rng = np.random.default_rng(12)
    for step in range(7):
        act = rng.integers(0, 29, size=(e, 3), dtype=np.uint8)
        ref.step(torch.from_numpy(act).cuda())
        out = dut.step_host(act, compact=True, chunks=(0, 3)[step & 1])
        assert np.array_equal(out["state32"].astype(np.int64), ref.state.cpu().numpy()[:, 0])
        assert np.array_equal(out["reward"], ref.reward.cpu().numpy())
        assert np.array_equal(out["done"], ref.terminated.cpu().numpy() | (ref.truncated.cpu().numpy() << 1))
    with pytest.raises(ValueError):
        _mk("pbn70", 1024).step_host(None, compact=True)
    ref.close()
    dut.close()


@pytest.mark.parametrize("name,e", [("pbn28", 5000), ("pbn10", 4096), ("pbn7", 1025)])
@pytest.mark.parametrize("chunks", [0, 3])
def test_packed_host_form_matches_oracle(name, e, chunks):
    """step_host(actions16=..., compact="packed"): 2 bytes up, one uint32 down per env.  Compared with the ORACLE
    (oracle.batched_step on the oracle's twin of the kernel's random streams), including the rewards the caller
    derives from reward_table()."""
    import torch
    from oracle import pbn_oracle as O
    from helpers import oracle_net
    net, onet = product_net(name), oracle_net(name)
    n = net.n_genes
    attrs = attractor_set(name)
    tables = O.attractor_tables(attrs.attractors, n)
    kw = dict(horizon=6, r_success=5.0, r_step=-0.25, r_action=-1.0)
    from pbn_rl_b200 import VecPBNEnv
    env = VecPBNEnv(net, e, attrs, device="cuda:0", perturb_p=0.01, perturb_mode="A", seed=77, **kw)
    _seed_env(env, name, e, 3)
    state = env.state.cpu().numpy().astype(np.uint64)
    target = env.target_id.cpu().numpy()
    t = np.zeros(e, dtype=np.uint16)
    rng = np.random.default_rng(4)
    table = env.reward_table()
    ids = np.arange(e, dtype=np.uint64)
    for step in range(4):
        act = rng.integers(0, n + 1, size=(e, 3), dtype=np.uint8)
        a16 = env.pinned_actions16()
        a16.numpy().view(np.uint16)[...] = env.pack_actions16(act)
        out = env.step_host(None, chunks=chunks, compact="packed", actions16=a16)
        if env.kernel == "sliced":
            sel, pert = O.sliced_stream(onet, 0.01, ids, step, 77)
        else:
            sel, pert = O.scalar_stream_selection(onet, ids, step, 77), O.scalar_stream_perturbation(n, 0.01, ids, step, 77)
        nxt, t, rew, term, trunc = O.batched_step(onet, tables, state, act, target, t, mode=O.PERT_A, sel=sel, pert=pert, **kw)
        packed = out["packed"]
        assert np.array_equal(packed & np.uint32((1 << 30) - 1), nxt[:, 0].astype(np.uint32)), f"state at step {step}"
        assert np.array_equal((packed >> np.uint32(30)) & np.uint32(1), term.astype(np.uint32))
        assert np.array_equal(packed >> np.uint32(31), trunc.astype(np.uint32))
        # rewards from the caller's own actions + the terminated bit
        nf = np.array([len({int(v) for v in row if 1 <= v <= n}) for row in act])
        assert np.array_equal(table[term.astype(np.int64), nf].view(np.uint32), rew.view(np.uint32))
        assert np.array_equal(env.reward.cpu().numpy().view(np.uint32), rew.view(np.uint32))
        state = nxt
    env.close()


@pytest.mark.parametrize("name,e", [("pbn28", 3000), ("pbn70", 2048)])
def test_step_host_matches_oracle(name, e):
    """The full-width host form against the oracle (not only against pbn_step)."""
    import torch
    from oracle import pbn_oracle as O
    from helpers import oracle_net
    net, onet = product_net(name), oracle_net(name)
    n = net.n_genes
    attrs = attractor_set(name)
    tables = O.attractor_tables(attrs.attractors, n)
    kw = dict(horizon=6, r_success=5.0, r_step=-0.25, r_action=-1.0)
    from pbn_rl_b200 import VecPBNEnv
    env = VecPBNEnv(net, e, attrs, device="cuda:0", perturb_p=0.01, perturb_mode="B", seed=77, **kw)
    _seed_env(env, name, e, 8)
    state = env.state.cpu().numpy().astype(np.uint64)
    target = env.target_id.cpu().numpy()
    t = np.zeros(e, dtype=np.uint16)
    rng = np.random.default_rng(6)
    ids = np.arange(e, dtype=np.uint64)
    for step in range(3):
        act = rng.integers(0, n + 1, size=(e, 3), dtype=np.uint8)
        out = env.step_host(act, chunks=2)
        sel, pert = O.sliced_stream(onet, 0.01, ids, step, 77)
        nxt, t, rew, term, trunc = O.batched_step(onet, tables, state, act, target, t, mode=O.PERT_B, sel=sel, pert=pert, **kw)
        assert np.array_equal(out["state"].astype(np.uint64), nxt)
        assert np.array_equal(out["reward"].view(np.uint32), rew.view(np.uint32))
        assert np.array_equal(out["terminated"], term) and np.array_equal(out["truncated"], trunc)
        state = nxt
    env.close()


_MODES = ["host_counter", "device_counter", "pdl"]


@pytest.mark.parametrize("mode,e", [pytest.param(m, (1 << 18) + 1024 + 7, id=m) for m in _MODES] +
                         [pytest.param(m, 5000, id=m + "-5000") for m in _MODES])
def test_packed_lane_form_and_graph_replay_equal_step(mode, e):
    """The packed form runs as lanes (each lane: upload -> unpack -> step -> export on its own stream); with a device
    step counter the whole step is captured on the second call with the same arguments and replayed as one graph launch
    from the third on.  Seven steps alternating two pinned action buffers must equal pbn_step on a twin env, step for
    step (eager, capture and replay calls all occur)."""
    import torch
    name = "pbn28"
    kw = dict(auto_reset=True)
    if mode != "host_counter":
        kw.update(device_counter=True, pdl=(mode == "pdl"))
    ref, dut = _mk(name, e, **kw), _mk(name, e, **kw)
    for env in (ref, dut):
        _seed_env(env, name, e, 11)
    rng = np.random.default_rng(12)
    bufs, acts = [], []
    for k in range(2):
        act = rng.integers(0, 29, size=(e, 3), dtype=np.uint8)
        b = torch.empty((e,), dtype=torch.int16, pin_memory=True)
        b.numpy().view(np.uint16)[...] = dut.pack_actions16(act)
        bufs.append(b)
        acts.append(torch.from_numpy(act).cuda())
    launches0 = dut.launches
    for step in range(7):
        out = dut.step_host(None, compact="packed", actions16=bufs[step % 2])
        ref.step(acts[step % 2])
        if mode == "pdl":
            ref.advance_counter()
        torch.cuda.synchronize()
        want = ref.state.cpu().numpy().astype(np.uint64)[:, 0].astype(np.uint32)
        packed = out["packed"]
        assert np.array_equal(packed & np.uint32((1 << 30) - 1), want), f"state at step {step}"
        assert np.array_equal((packed >> np.uint32(30)) & np.uint32(1), ref.terminated.cpu().numpy().astype(np.uint32))
        assert np.array_equal(packed >> np.uint32(31), ref.truncated.cpu().numpy().astype(np.uint32))
    per_step = (dut.launches - launches0) / 7
    # lanes x (unpack, step, export), + the counter update with a device counter; from 2^18 envs on 2 lanes, 4 when the
    # step is replayed as a graph (device counter): 13 / 6 launches per step at 2^18 + 1031 envs
    lanes = 1 if e < (1 << 18) else (2 if mode == "host_counter" else 4)
    assert per_step == lanes * 3 + (1 if mode != "host_counter" else 0)
    assert np.array_equal(dut.state.cpu().numpy(), ref.state.cpu().numpy())
    ref.close(); dut.close()


@pytest.mark.parametrize("compact", [False, True, "packed"])
def test_step_host_between_pdl_steps(compact):
    """On a pdl env, step_host closes the open PDL sequence and the library advances the device counter itself:
    steps and host steps interleaved (two host steps in a row included) draw the random streams of a host-counter twin,
    step for step."""
    import torch
    e, name = 3 * 1024 + 5, "pbn28"
    ref = _mk(name, e, auto_reset=True)
    dut = _mk(name, e, auto_reset=True, pdl=True)
    for env in (ref, dut):
        _seed_env(env, name, e, 13)
    rng = np.random.default_rng(14)
    a16 = dut.pinned_actions16()
    for step in range(8):
        act = rng.integers(0, 29, size=(e, 3), dtype=np.uint8)
        ref.step(torch.from_numpy(act).cuda())
        state, term, trunc = (x.cpu().numpy() for x in (ref.state, ref.terminated, ref.truncated))
        reward = ref.reward.cpu().numpy()
        if step not in (2, 3, 6):
            dut.step(torch.from_numpy(act).cuda())
            assert np.array_equal(dut.state.cpu().numpy(), state), f"state at step {step}"
            assert np.array_equal(dut.reward.cpu().numpy(), reward), f"reward at step {step}"
            continue
        if compact == "packed":
            a16.numpy().view(np.uint16)[...] = dut.pack_actions16(act)
            out = dut.step_host(None, compact="packed", actions16=a16)
            packed = out["packed"]
            assert np.array_equal(packed & np.uint32((1 << 30) - 1), state[:, 0].astype(np.uint32)), f"state at step {step}"
            assert np.array_equal((packed >> np.uint32(30)) & np.uint32(1), term.astype(np.uint32))
            assert np.array_equal(packed >> np.uint32(31), trunc.astype(np.uint32))
        elif compact:
            out = dut.step_host(act, compact=True)
            assert np.array_equal(out["state32"].astype(np.int64), state[:, 0]), f"state at step {step}"
            assert np.array_equal(out["reward"], reward)
            assert np.array_equal(out["done"], term | (trunc << 1))
        else:
            out = dut.step_host(act)
            assert np.array_equal(out["state"], state), f"state at step {step}"
            assert np.array_equal(out["reward"], reward)
            assert np.array_equal(out["terminated"], term) and np.array_equal(out["truncated"], trunc)
    dut.advance_counter()
    assert int(dut.step_ctr_dev.item()) == 8
    assert ref.stats() == dut.stats()
    ref.close(); dut.close()


def test_packed_graph_cache_survives_more_buffers_than_slots():
    """Ten distinct pinned action buffers against the library's eight graph slots: entries are evicted and captured
    again, every call still returns what pbn_step returns."""
    import torch
    name, e = "pbn28", 1 << 18
    ref, dut = _mk(name, e, auto_reset=True, device_counter=True), _mk(name, e, auto_reset=True, device_counter=True)
    for env in (ref, dut):
        _seed_env(env, name, e, 21)
    rng = np.random.default_rng(22)
    bufs, acts = [], []
    for k in range(10):
        act = rng.integers(0, 29, size=(e, 3), dtype=np.uint8)
        b = torch.empty((e,), dtype=torch.int16, pin_memory=True)
        b.numpy().view(np.uint16)[...] = dut.pack_actions16(act)
        bufs.append(b)
        acts.append(torch.from_numpy(act).cuda())
    for step in range(25):
        k = (step * 7) % 10 if step >= 10 else step
        out = dut.step_host(None, compact="packed", actions16=bufs[k])
        ref.step(acts[k])
        torch.cuda.synchronize()
        want = ref.state.cpu().numpy().astype(np.uint64)[:, 0].astype(np.uint32)
        assert np.array_equal(out["packed"] & np.uint32((1 << 30) - 1), want), f"state at step {step}"
    assert dut.stats() == ref.stats()   # episode statistics accumulated on the device by both paths
    ref.close(); dut.close()
