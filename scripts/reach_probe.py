"""Exhaustive attractor search (find_attractors_exhaustive, pbn_reach_sweep): what it finds and what it costs.

On Bittner-28, make_network(20, 3, 4, seed=20) and make_network(24, 2, 3, seed=24) with the default arguments, then on
the 20-gene network again with a closure limit of 2^20 states:
1. End-to-end wall time of find_attractors_exhaustive (default arguments), a first call (including the run-time
   specialisation of the rollout kernel) and a second one; attractors, sweeps, rounds, how many the rollout seeding found.
2. CUDA-event device time of every sweep from the states of all attractors to the fixed point, and of one more sweep
   once every state is marked (the skip pass).
3. The states that cannot reach a marked state: all attractors but the one with the largest sampled basin are marked and
   swept to the fixed point; then one more sweep marks nothing and its time is the cost of those states alone.
4. Bittner-28 only: one pbn_dp_expect at p = 0, for comparison with a sweep.
Writes <out>/r08_reach_probe.json; the card's name and power limit are read in the same run.

    python scripts/reach_probe.py [--out profiles]
"""
import argparse
import json
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "tests"), str(ROOT / "scripts")]

from control_probe import card, timed  # noqa: E402


def event_time(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3, out


def sweep_times(env, seeds):
    """Mark ``seeds``, then sweep to the fixed point: [(device seconds, states marked)] per sweep."""
    from pbn_rl_b200.discover import ReachMarks
    reach = ReachMarks(env)
    reach.mark(seeds)
    out = []
    while True:
        t, k = event_time(reach.sweep)   # sweep() reads the count back, after the event pair
        out.append((t, k))
        if k == 0:
            return out, reach


def case(name, net, **kw):
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200.discover import find_attractors_exhaustive, find_attractors_rollout
    rec = {"case": name, "n_genes": net.n_genes, "args": kw}
    for tag in ("first", "warm"):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, info = find_attractors_exhaustive(net, **kw)
        torch.cuda.synchronize()
        rec["wall_s_%s" % tag] = time.perf_counter() - t0
    states = info.pop("states")
    rec.update(info)
    rec["attractors"] = len(states)
    rec["attractor_sizes"] = sorted(len(m) for m in states)
    _, rinfo = find_attractors_rollout(net)
    rec["rollout_attractors"] = len(rinfo["states"])
    rec["rollout_missed"] = len({tuple(m) for m in states} - {tuple(m) for m in rinfo["states"]})

    env = VecPBNEnv(net, 1024, None, device="cuda:0", horizon=0, bins=1, perturb_p=0.0)
    full, reach = sweep_times(env, [s for m in states for s in m])
    rec["cover_sweeps"] = [{"s": t, "marked": k} for t, k in full]
    rec["cover_device_s"] = sum(t for t, _ in full)
    rec["covered"] = reach.count
    rec["skip_sweep_s"] = timed(reach.sweep)[0]
    if len(states) > 1:
        big = max(range(len(rinfo["states"])), key=lambda i: rinfo["basin_fraction"][i])
        left = rinfo["states"][big]
        part, reach = sweep_times(env, [s for m in states if m != left for s in m])
        rec["left_out_size"] = len(left)
        rec["left_out_uncovered"] = reach.uncovered
        rec["partial_cover_device_s"] = sum(t for t, _ in part)
        rec["stuck_sweep_s"] = timed(reach.sweep, max_reps=5)[0]
    env.close()
    if net.n_genes == 28:
        from pbn_rl_b200.control import _Backup
        env = VecPBNEnv(net, 1, None, device="cuda:0", perturb_p=0.0, kernel="scalar")
        bk = _Backup(env)
        u = torch.randn(1 << 28, dtype=torch.float64, device="cuda:0")
        rec["dp_expect_s"] = event_time(lambda: bk.expect(u))[0]
        env.close()
        del bk, u
        torch.cuda.empty_cache()
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles"))
    args = ap.parse_args()
    from helpers import make_network, product_net
    from pbn_rl_b200 import PBNNetwork
    pbn28 = product_net("pbn28")
    net20 = PBNNetwork.from_expressions(*make_network(20, 3, 4, seed=20))
    net24 = PBNNetwork.from_expressions(*make_network(24, 2, 3, seed=24))
    runs = [("Bittner-28", pbn28, {}), ("make_network(20, 3, 4, seed=20)", net20, {}),
            ("make_network(24, 2, 3, seed=24)", net24, {}),
            ("make_network(20, 3, 4, seed=20)", net20, {"max_attractor_states": 1 << 20})]
    out = {"card": card(), "torch": torch.__version__, "cases": []}
    Path(args.out).mkdir(parents=True, exist_ok=True)
    for name, net, kw in runs:   # the file is rewritten after every case
        out["cases"].append(case(name, net, **kw))
        (Path(args.out) / "r08_reach_probe.json").write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
