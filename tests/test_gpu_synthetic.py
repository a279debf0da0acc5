"""GPU: randomly generated networks at the edges of what the ABI admits -- 1 gene, exactly 32 / 64 / 96 / 128
genes, 1..5 predictors per gene, arities 0..9 (constants, wide predictors), 1..8 action slots, wildcard targets --
against the oracle, which parses the same expression strings with its own evaluator."""
import numpy as np
import pytest

from helpers import CASES, make_attractors, make_network

pytestmark = pytest.mark.gpu

MODES = {"none": 0, "A": 1, "B": 2, "C": 3}


@pytest.mark.parametrize("n,kmax,amax,bins,uniform,kernels", CASES)
@pytest.mark.parametrize("mode", ["A", "C"])
def test_synthetic_networks_bit_exact(n, kmax, amax, bins, uniform, kernels, mode):
    import torch
    from oracle import pbn_oracle as O
    from pbn_rl_b200 import AttractorSet, PBNNetwork, VecPBNEnv
    genes, exprs = make_network(n, kmax, amax, seed=1000 + n)
    net = PBNNetwork.from_expressions(genes, exprs)
    onet = O.OracleNetwork(genes, exprs)
    attrs = make_attractors(n, 5, seed=n)
    aset = AttractorSet(attrs, n)
    tables = O.attractor_tables(attrs, n)
    e, p, seed = 1500, 0.03, 4242
    rng = np.random.default_rng(n)
    w = net.n_words
    masks = np.array(net.state_mask(), dtype=np.uint64)
    state0 = ((rng.integers(0, 2**63, size=(e, w), dtype=np.int64).astype(np.uint64) * np.uint64(2))
              + rng.integers(0, 2, size=(e, w)).astype(np.uint64)) & masks
    target = rng.integers(-1, 5, size=e).astype(np.int32)
    kw = dict(horizon=3, r_success=2.5, r_step=-0.5, r_action=-1.0)
    for kernel in kernels:
        env = VecPBNEnv(net, e, aset, device="cuda:0", perturb_p=p, perturb_mode=mode, seed=seed, bins=bins, kernel=kernel, **kw)
        assert env.kernel == kernel
        env.set_state(torch.from_numpy(state0.astype(np.int64)), packed=True)
        env.set_target(torch.from_numpy(target))
        state, t = state0, np.zeros(e, np.uint16)
        ids = np.arange(e, dtype=np.uint64)
        for step in range(3):
            act = rng.integers(0, n + 1, size=(e, bins), dtype=np.uint8)
            if step == 1:      # injected randomness
                sel = np.stack([rng.integers(0, len(r), size=e) for r in exprs], axis=1).astype(np.uint8)
                pert = (rng.integers(0, 2**63, size=(e, w), dtype=np.int64).astype(np.uint64) & masks) * (rng.random((e, 1)) < 0.3)
                pert = pert.astype(np.uint64)
                env.step_injected(torch.from_numpy(act), torch.from_numpy(sel), torch.from_numpy(pert.astype(np.int64)))
                env.step_ctr = step + 1
            else:
                env.step(torch.from_numpy(act).cuda())
                if kernel == "scalar":
                    sel = O.scalar_stream_selection(onet, ids, step, seed)
                    pert = O.scalar_stream_perturbation(n, p, ids, step, seed)
                else:
                    sel, pert = O.sliced_stream(onet, p, ids, step, seed)
            nxt, t1, rew, term, trunc = O.batched_step(onet, tables, state, act, target, t, mode=MODES[mode], sel=sel, pert=pert, **kw)
            torch.cuda.synchronize()
            tag = "n=%d %s %s step %d" % (n, kernel, mode, step)
            assert np.array_equal(env.state.cpu().numpy().astype(np.uint64), nxt), tag
            assert np.array_equal(env.reward.cpu().numpy(), rew), tag
            assert np.array_equal(env.terminated.cpu().numpy(), term) and np.array_equal(env.truncated.cpu().numpy(), trunc), tag
            assert np.array_equal(env.t.cpu().numpy().astype(np.uint16), t1), tag
            state, t = nxt, t1
        if kernel == "sliced":      # uncontrolled rollout on the same odd-shaped network
            ref = env.state.clone()
            twin = VecPBNEnv(net, e, aset, device="cuda:0", perturb_p=p, perturb_mode=mode, seed=seed, bins=bins, kernel=kernel, **kw)
            twin.set_state(ref, packed=True)
            twin.step_ctr = env.step_ctr
            for _ in range(4):
                twin.step(None)
            env.rollout(4)
            assert torch.equal(env.state, twin.state), "rollout n=%d %s" % (n, mode)
            twin.close()
        env.close()
