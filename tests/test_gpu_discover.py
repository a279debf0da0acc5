"""GPU: attractor discovery by massive rollouts + device visit-count hash (pbn_rl_b200/discover.py)
against the known answers K2/K5 (tests/golden/k5_stg.json: sink SCCs of pbn7/pbn10 by brute force) and,
for the large networks, against closure/connectivity checks done with the oracle's evaluator."""
import numpy as np
import pytest

from helpers import golden, oracle_net, product_net

pytestmark = pytest.mark.gpu


def _oracle_descriptor(onet, s):
    """(can1, can0) of state s from the oracle: OR over 'every gene uses its predictor min(k, K_i - 1)'."""
    can1 = can0 = 0
    full = (1 << onet.n) - 1
    nf = [len(row) for row in onet.py_code]
    for k in range(max(nf)):
        t = onet.transition(s, 0, [min(k, nf[i] - 1) for i in range(onet.n)], 0)
        can1 |= t
        can0 |= ~t & full
    return can1, can0


def _successors(can1, can0):
    free = can1 & can0
    out = [can1 & ~free]
    b = free
    while b:
        low = b & -b
        out += [t | low for t in out]
        b ^= low
    return out


@pytest.mark.parametrize("method", ["device", "host"])
@pytest.mark.parametrize("name", ["pbn7", "pbn10"])
def test_rollout_finder_reproduces_brute_force_sink_sccs(name, method):
    from pbn_rl_b200.discover import find_attractors_rollout
    attrs, info = find_attractors_rollout(product_net(name), n_rollouts=4096, burn_in=200, method=method)
    want = golden("k5_stg.json")[name]["sink_sccs"]
    assert info["states"] == [sorted(m) for m in sorted(want, key=lambda m: min(m))]
    assert abs(sum(info["basin_fraction"]) - 1.0) < 1e-9 and not info["unresolved"]
    assert len(attrs) == len(want)


@pytest.mark.parametrize("name,kernel", [("pbn7", "auto"), ("pbn10", "scalar")])
def test_successor_sets_match_host_enumeration(name, kernel):
    import torch
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200.attractors import _successor_sets
    from pbn_rl_b200.discover import successor_descriptors
    net = product_net(name)
    env = VecPBNEnv(net, 1024, None, device="cuda:0", kernel=kernel)
    can1, can0 = _successor_sets(net)
    got = successor_descriptors(env, list(range(1 << net.n_genes)))
    assert [g[0] for g in got] == can1.tolist() and [g[1] for g in got] == can0.tolist()
    env.close()


@pytest.mark.parametrize("name", ["pbn28", "pbn70"])
def test_large_network_attractors_are_closed_and_strongly_connected(name):
    from pbn_rl_b200.discover import find_attractors_rollout
    onet = oracle_net(name)
    attrs, info = find_attractors_rollout(product_net(name), n_rollouts=1 << 14, burn_in=300, max_candidates=64)
    if name == "pbn28":   # the host closure + Tarjan path finds the very same attractors
        _, info_host = find_attractors_rollout(product_net(name), n_rollouts=1 << 14, burn_in=300, max_candidates=64,
                                               method="host")
        assert info_host["states"] == info["states"]
    assert len(attrs) >= 1 and sum(info["basin_fraction"]) > 0.5
    for members in info["states"][:12]:
        mset = set(members)
        succ = {}
        for s in members[:64]:
            succ[s] = _successors(*_oracle_descriptor(onet, s))
            assert set(succ[s]) <= mset, "attractor is not closed under the oracle's transition relation"
        if len(members) <= 64:           # strongly connected: everything reaches the first member and back
            reach = {members[0]}
            todo = [members[0]]
            while todo:
                for t in succ[todo.pop()]:
                    if t not in reach:
                        reach.add(t)
                        todo.append(t)
            assert reach == mset


@pytest.mark.parametrize("name,e", [("pbn10", 5000), ("pbn70", 3000)])
def test_visit_count_equals_numpy_unique(name, e):
    import torch
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200.discover import VisitCounter
    net = product_net(name)
    env = VecPBNEnv(net, e, None, device="cuda:0")
    rng = np.random.default_rng(3)
    table = VisitCounter(env, 1 << 12)
    ref = {}
    for rnd in range(3):
        st = rng.integers(0, 40, size=(e, net.n_words), dtype=np.int64)     # many duplicates
        if net.n_words == 2:
            st[:, 1] = rng.integers(0, 3, size=e)
        mask = (rng.random(e) < 0.7).astype(np.uint8) if rnd else None
        table.add(torch.from_numpy(st), None if mask is None else torch.from_numpy(mask))
        for k in range(e):
            if mask is None or mask[k]:
                key = tuple(int(x) for x in st[k])
                ref[key] = ref.get(key, 0) + 1
    states, counts = table.items()
    got = {tuple(int(x) for x in states[k]): int(counts[k]) for k in range(len(counts))}
    assert got == ref
    small = VisitCounter(env, 16)                                            # too small: overflow is reported
    small.add(torch.arange(e, dtype=torch.int64).reshape(e, 1).repeat(1, net.n_words))
    with pytest.raises(RuntimeError):
        small.items()
    env.close()


def test_steady_state_histogram_mass():
    import torch
    from helpers import attractor_set
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200.discover import steady_state_histogram
    net = product_net("pbn7")
    env = VecPBNEnv(net, 2048, None, device="cuda:0", perturb_p=0.0)
    env.state.random_(0, 128)
    hist = steady_state_histogram(env, steps=20, burn_in=200)
    assert sum(hist.values()) == 20 * 2048
    sinks = {s for m in golden("k5_stg.json")["pbn7"]["sink_sccs"] for s in m}
    assert set(hist) <= sinks                    # without perturbation all mass sits on the attractors
    proj = steady_state_histogram(env, steps=5, genes=[0, 6])
    assert sum(proj.values()) == 5 * 2048 and set(proj) <= {0, 1, 2, 3}
    env.close()


def test_basin_labels_match_exhaustive_reachability():
    """pbn10 without perturbation: every state is labelled with an attractor it can reach in the brute-force STG
    (K5), and states inside an attractor are labelled with it after 0 steps."""
    import torch
    from pbn_rl_b200 import AttractorSet, VecPBNEnv
    from pbn_rl_b200.attractors import _successor_sets, _successors
    from pbn_rl_b200.discover import basin_labels
    net = product_net("pbn10")
    sinks = golden("k5_stg.json")["pbn10"]["sink_sccs"]
    aset = AttractorSet([[tuple((s >> i) & 1 for i in range(10)) for s in m] for m in sinks], 10)
    env = VecPBNEnv(net, 1024, aset, device="cuda:0", perturb_p=0.0)
    env.set_state(torch.arange(1024, dtype=torch.int64).reshape(-1, 1), packed=True)
    ids, steps = basin_labels(env, max_steps=512)
    ids, steps = ids.cpu().numpy(), steps.cpu().numpy()
    assert (ids >= 0).all()
    can1, can0 = _successor_sets(net)
    succ = [_successors(s, int(can1[s]), int(can0[s]), 10) for s in range(1024)]
    reach = []                                   # attractors reachable from each state (backward closure per attractor)
    pred = [[] for _ in range(1024)]
    for s in range(1024):
        for t in succ[s]:
            pred[t].append(s)
    for m in sinks:
        seen, todo = set(m), list(m)
        while todo:
            for q in pred[todo.pop()]:
                if q not in seen:
                    seen.add(q)
                    todo.append(q)
        reach.append(seen)
    for s in range(1024):
        assert s in reach[ids[s]], s
    for a, m in enumerate(sinks):
        for s in m:
            assert ids[s] == a and steps[s] == 0
    env.close()


def test_bench_runs_on_a_small_configuration():
    """bench.py end to end (tiny batch): exactly one JSON line on stdout with the contract's keys."""
    import json
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    out = subprocess.run([sys.executable, str(root / "bench.py"), "--envs", "8192", "--batches", "2", "--steps", "10", "--warmup", "3",
                          "--no-cpu-baseline", "--no-configs", "--strong", "--e2e-steps", "2"], capture_output=True, text=True, timeout=600, cwd=str(root))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert key in d, key
    assert d["steps"] == 10 and d["gpu_launches"] == 10 and d["value"] > 0 and d["roofline"]["bound"] == "hbm"
    assert d["e2e"]["h2d_bytes_per_step"] == 8192 * 2 and d["e2e"]["d2h_bytes_per_step"] == 8192 * 4   # packed host form
    assert d["strong"]["total_envs"] == 8192 and d["strong"]["value"] > 0 and d["configs"] is None


def test_bench_dumps_the_same_outputs_from_run_to_run(tmp_path):
    """bench.py --dump-outputs: the last timed step's results, identical for identical arguments; --steps is the number
    of timed steps also when it is not a multiple of the graph length."""
    import json
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, str(root / "bench.py"), "--envs", "8192", "--batches", "2", "--steps", "7",
                              "--graph-steps", "4", "--warmup", "3", "--no-cpu-baseline", "--no-configs", "--e2e-steps", "2",
                              "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600, cwd=str(root))
        assert out.returncode == 0, out.stderr[-2000:]
        d = json.loads(out.stdout)
        assert d["steps"] == 7 and d["gpu_launches"] == 7
        dumps.append({p.stem: np.load(p) for p in (tmp_path / run).glob("*.npy")})
    a, b = dumps
    assert sorted(a) == ["reward", "state_u32", "terminated", "truncated"]
    assert a["state_u32"].shape == (8192, 2) and a["state_u32"].dtype == np.float64
    assert a["state_u32"][:, 0].max() < 2**28 and not a["state_u32"][:, 1].any()   # 28-gene states
    assert a["state_u32"][:, 0].any() and a["reward"].any()
    assert set(np.unique(a["terminated"])) <= {0.0, 1.0} and set(np.unique(a["truncated"])) <= {0.0, 1.0}
    for name in a:
        assert np.array_equal(a[name], b[name]), name
