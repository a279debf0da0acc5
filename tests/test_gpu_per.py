"""GPU: prioritised replay on the device (pbn_per_*, DevicePrioritizedReplay) against the float32 restatement of its
contract (oracle/per_oracle.py)."""
import numpy as np
import pytest

from helpers import attractor_set, product_net
from oracle import per_oracle as P

pytestmark = pytest.mark.gpu


def _env(name, e):
    import torch
    from pbn_rl_b200 import VecPBNEnv
    env = VecPBNEnv(product_net(name), e, attractor_set(name), device="cuda:0", horizon=5, bins=3, perturb_p=0.02,
                    perturb_mode="A", seed=3, auto_reset=True)
    env.reset()
    torch.cuda.synchronize()
    return env


def _within_ulps(a, b, k):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return np.all(np.abs(a.astype(np.float64) - b) <= k * np.spacing(np.maximum(np.abs(a), np.abs(b))))


def _check_tree(ring, orc):
    """Leaves within 2 ulp of the oracle (device powf is not correctly rounded); every stored node, total and pmin
    bit-identical to the oracle trees rebuilt from the device's own leaves; max_p exact.  Re-syncs the oracle."""
    import torch
    torch.cuda.synchronize()
    L, cap = ring.leaves_pow2, ring.capacity
    leaves = ring.leaves().cpu().numpy()
    min_leaves = ring.levels()[0][1][:cap].cpu().numpy()
    assert _within_ulps(leaves, orc.leaves(), 2)
    unwritten = np.isinf(orc.m[L:L + cap])          # +inf in the min tree, 0 in the sum tree
    assert np.array_equal(np.isinf(min_leaves), unwritten)
    assert np.array_equal(min_leaves[~unwritten], leaves[~unwritten]) and not leaves[unwritten].any()
    s, m = P.build_trees(leaves, min_leaves, L)
    P.rebuild(s, m, L)
    n = L
    for got_s, got_m in ring.levels():
        assert np.array_equal(got_s.cpu().numpy(), s[n:2 * n]), n
        assert np.array_equal(got_m.cpu().numpy(), m[n:2 * n]), n
        n //= 2
    assert ring.total() == s[1] and ring.pmin() == m[1]
    assert np.float32(ring.max_p()) == orc.max_p
    orc.s[:], orc.m[:] = s, m
    return s, m


def _check_sample(ring, s, m, batch, seed, beta=0.4):
    import torch
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    u = torch.rand((batch,), device="cuda:0", generator=g)
    u[-1] = float(np.nextafter(np.float32(1), np.float32(0)))   # a mass that can round up to total
    out = ring.sample(batch, beta=beta, u=u)
    torch.cuda.synchronize()
    want_i, want_w = P.sample(s, m, ring.leaves_pow2, u.cpu().numpy(), beta)
    got_i = out["index"].cpu().numpy()
    assert np.array_equal(got_i, want_i)
    assert np.all(got_i < ring.size)
    w = out["weight"].cpu().numpy()
    assert w.shape == (batch, 1) and np.allclose(w[:, 0], want_w, rtol=1e-5, atol=0)
    plain = super(type(ring), ring).sample(batch, index=out["index"])
    for key in ("obs", "next_obs", "actions", "reward", "done"):
        assert torch.equal(out[key], plain[key]), key
    return out


@pytest.mark.parametrize("name,e,cap", [("pbn7", 37, 100), ("pbn28", 1500, 4000), ("pbn70", 300, 700), ("pbn10", 64, 64)])
def test_trees_and_samples_match_the_oracle(name, e, cap):
    import torch
    from pbn_rl_b200.replay import DevicePrioritizedReplay
    env = _env(name, e)
    ring = DevicePrioritizedReplay(env, cap, alpha=0.6, eps=1e-6)
    orc = P.OraclePER(cap, 0.6)
    rng = np.random.default_rng(11)
    n = env.n_genes
    for step in range(7):   # wraps the ring for every case
        head = ring.head
        ring.step(torch.from_numpy(rng.integers(0, n + 1, size=(e, 3), dtype=np.uint8)).cuda())
        orc.push(head, e)
        s, m = _check_tree(ring, orc)
        if step == 0:
            _check_sample(ring, s, m, 256, seed=step)       # partly filled ring (except capacity == num_envs)
        for b in (1, 257, 5000):                            # 5000: the multi-CTA update
            idx = rng.integers(0, ring.size, size=b)
            if b > 1:
                idx[rng.integers(0, b, size=b // 8)] = idx[0]              # duplicates
                idx[rng.integers(0, b, size=3)] = [-1, cap, cap + 17]      # ignored
            td = (rng.standard_normal(b) * rng.exponential(3.0, b)).astype(np.float32)
            if b > 1:
                td[:2] = [np.nan, np.inf]
            ring.update_priorities(torch.from_numpy(idx).cuda(), torch.from_numpy(td).cuda())
            orc.update(idx, td, 1e-6)
            s, m = _check_tree(ring, orc)
    for batch in (1, 256, 4096):
        _check_sample(ring, s, m, batch, seed=batch)
    env.close()


def test_duplicates_range_clamp_and_max_p():
    import torch
    from pbn_rl_b200 import _cabi
    from pbn_rl_b200.replay import DevicePrioritizedReplay
    env = _env("pbn10", 64)
    ring = DevicePrioritizedReplay(env, 100, alpha=0.5, eps=0.25)
    orc = P.OraclePER(100, 0.5)
    assert ring.max_p() == 1.0 and ring.total() == 0.0 and ring.pmin() == float("inf")
    dev = lambda a, dt=torch.int64: torch.tensor(a, dtype=dt, device="cuda:0")

    def update(idx, td):
        ring.update_priorities(dev(idx), dev(td, torch.float32))
        orc.update(idx, np.array(td, dtype=np.float32), 0.25)
        _check_tree(ring, orc)
        return ring.leaves().cpu().numpy()

    l0 = env.launches
    ring.push(90, 20)                                    # wraps: 90..99, 0..9
    orc.push(90, 20)
    assert env.launches == l0 + 1                        # one launch per push
    assert ring.leaves().cpu().tolist() == [1.0] * 10 + [0.0] * 80 + [1.0] * 10
    _check_tree(ring, orc)
    l0 = env.launches
    lv = update([5, 5, 5], [3.75, 15.75, 0.0])
    assert env.launches == l0 + 1                        # small batches: one CTA, one launch
    assert lv[5] == 0.5                                  # the last occurrence: sqrt(0 + 0.25)
    assert ring.max_p() == 16.0                          # every valid entry folds into max_p
    before = ring.tree.clone()
    update([-1, 100, 1 << 40], [1e6, 1e6, 1e6])          # outside [0, capacity): ignored
    assert torch.equal(ring.tree.view(torch.int32), before.view(torch.int32)) and ring.max_p() == 16.0
    lv = update([6, 7, 8], [float("nan"), float("inf"), -float("inf")])
    assert lv[6] == 0.5 and lv[7] == lv[8] and _within_ulps(lv[7], np.float32(1e15), 2)
    assert ring.max_p() == np.float32(1e30)
    assert np.isfinite(ring.tree[1:2 * ring.leaves_pow2].cpu().numpy()).all()
    update([7, 8], [0.0, 0.0])
    assert ring.max_p() == np.float32(1e30)              # never decreases
    ring.push(20, 1)                                     # enters at max_p ** alpha
    orc.push(20, 1)
    _check_tree(ring, orc)
    assert _within_ulps(ring.leaves()[20].item(), np.float32(1e15), 2)
    with pytest.raises(ValueError):
        DevicePrioritizedReplay(env, 100, eps=0.0)
    with pytest.raises(_cabi.PbnError):
        ring.push(100, 1)
    env.close()


def test_large_ring_distribution():
    """capacity 2^22, one push of 2^20, every pushed priority updated at random (the multi-CTA update): the tree is
    exact and the sampled slot buckets follow the leaf masses."""
    import torch
    from scipy.stats import chisquare

    from pbn_rl_b200.replay import DevicePrioritizedReplay
    env = _env("pbn10", 64)
    ring = DevicePrioritizedReplay(env, 1 << 22)
    n = 1 << 20
    ring.push(0, n)
    ring.size = n
    g = torch.Generator(device="cuda:0").manual_seed(5)
    idx = torch.randperm(n, device="cuda:0", generator=g)
    td = torch.rand((n,), device="cuda:0", generator=g) * 4.0
    ring.update_priorities(idx, td)
    orc = P.OraclePER(1 << 22, 0.6)
    orc.push(0, n)
    orc.update(idx.cpu().numpy(), td.cpu().numpy(), 1e-6)
    s, m = _check_tree(ring, orc)
    _check_sample(ring, s, m, 4096, seed=9)
    buckets = 64
    counts = np.zeros(buckets)
    for k in range(64):
        out = ring.sample(4096, generator=g)
        counts += np.bincount(out["index"].cpu().numpy() * buckets // n, minlength=buckets)
    mass = ring.leaves()[:n].double().reshape(buckets, -1).sum(1).cpu().numpy()
    assert chisquare(counts, counts.sum() * mass / mass.sum()).pvalue > 1e-4
    env.close()


def test_cuda_graph_replay_equals_eager():
    import torch
    from pbn_rl_b200.replay import DevicePrioritizedReplay
    env = _env("pbn28", 1024)
    ring = DevicePrioritizedReplay(env, 3000)
    for _ in range(3):
        ring.step(None)
    g = torch.Generator(device="cuda:0").manual_seed(1)
    u = torch.rand((256,), device="cuda:0", generator=g)
    td = torch.randn((256,), device="cuda:0", generator=g)
    torch.cuda.synchronize()
    tree0, maxp0 = ring.tree.clone(), ring.max_p_buf.clone()

    def seq():
        out = ring.sample(256, beta=0.5, u=u)
        ring.update_priorities(out["index"], td * out["weight"][:, 0])
        return out

    eager = seq()
    torch.cuda.synchronize()
    eager = {k: v.clone() for k, v in eager.items()}
    tree1, maxp1 = ring.tree.clone(), ring.max_p_buf.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):      # warm-up on the capture stream
        seq()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = seq()
    ring.tree.copy_(tree0)
    ring.max_p_buf.copy_(maxp0)
    graph.replay()
    torch.cuda.synchronize()
    for k, v in eager.items():
        assert torch.equal(static[k], v), k
    # bit patterns: the scratch words at the end of the tree array are int32 (-1 reads as a float NaN)
    assert torch.equal(ring.tree.view(torch.int32), tree1.view(torch.int32)) and torch.equal(ring.max_p_buf, maxp1)
    env.close()


def test_insitu_bdq_per_runs():
    import importlib.util
    from pathlib import Path
    spec = importlib.util.spec_from_file_location("insitu_bdq", Path(__file__).resolve().parent.parent / "scripts" / "insitu_bdq.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.run("pbn28", envs=4096, iters=4, warmup=1, batch=64, per=True)
    assert np.isfinite(out["loss_last"]) and out["per"]["weight_max"] <= 1.0 and out["per"]["total"] > 0
    assert out["phase_ms_per_iteration"]["per_push"] > 0 and out["phase_ms_per_iteration"]["per_update"] > 0
