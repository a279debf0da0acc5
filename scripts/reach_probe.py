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

--wide: above 28 genes, where the bitset (1 GiB at 33 genes, 2 GiB at 34) no longer fits the L2.  Bittner-28 again as
the reference, bb33 (33 genes, one predictor per gene) and trap_network(34) (tests/test_gpu_reach_wide.py: three of its
six attractors have basins of one or two states, which the seeding rollouts miss).  Steps 1, 2 and 4 as above, plus the
first sweep's device time per state; step 3 is left out, since at 34 genes it would sweep a quarter of the states
that walk their whole successor sets, several times.  Writes <out>/r09_reach_wide_probe.json.

--closure bitset: the search with closure="bitset" (pbn_reach_forward, attractor_in_closure).  make_network(20, 3, 4,
seed=20) with the hash and the bitset closure at a limit of 2^20 states and with the bitset closure at the default
limit; free-block networks (tests/reach_forward_oracle.py) with 18 free genes at 20 and 34 genes (at 34 also with genes
32 and 33 in the block) and with 22 at 34 genes; Bittner-28 and bb33 with both closures, alternated twice, and
trap_network(34) with both closures once.
Step 1 as above, with the forward and backward sweep counts of the attractor searches; then for one state of the
largest attractor, the CUDA-event device time of every forward sweep of its closure and of the sink test.  Writes
<out>/r10_reach_forward_probe.json.

    python scripts/reach_probe.py [--out profiles] [--wide | --closure bitset]
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


def case(name, net, partial=True, **kw):
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
    rec["first_sweep_ns_per_state"] = full[0][0] / (1 << net.n_genes) * 1e9
    rec["covered"] = reach.count
    rec["skip_sweep_s"] = timed(reach.sweep)[0]
    if partial and len(states) > 1:
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


def closure_profile(net, s):
    """Device time of each forward sweep from ``s`` to the fixed point, and of the sink test (bitwise not, mark, backward
    sweeps to the fixed point)."""
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200._cabi import check
    from pbn_rl_b200.discover import ReachMarks, _ForwardWorkspace
    env = VecPBNEnv(net, 1024, None, device="cuda:0", horizon=0, bins=1, perturb_p=0.0)
    ws = _ForwardWorkspace(env)
    lib, h, st = env.lib, env._h, env._stream()
    rec = {"state": s}
    ws.set.zero_()
    ws.done.zero_()
    ws._mark(ws.set, s)
    sweeps, size = [], 1

    def fwd():
        ws.newly.zero_()
        check(lib.pbn_reach_forward(h, ws.set.data_ptr(), ws.done.data_ptr(), ws.newly.data_ptr(), st))
    while True:
        t, _ = event_time(fwd)
        r, e = ws.newly.tolist()
        sweeps.append({"s": t, "reached": r, "expanded": e})
        size += r
        if e == 0:
            break
    rec.update(size=size, forward_sweeps=sweeps, forward_device_s=sum(x["s"] for x in sweeps))

    def sink_test():
        ws.done.bitwise_not_()
        ws._mark(ws.done, s)
        test = ReachMarks(env, marks=ws.done, count=(1 << net.n_genes) - size + 1)
        test.close()
        return test
    t, test = event_time(sink_test)
    rec.update(sink_test_s=t, sink_test_sweeps=test.sweeps, strongly_connected=test.uncovered == 0)
    env.close()
    del ws
    torch.cuda.empty_cache()
    return rec


def forward_case(name, net, kw, profile=True):
    from pbn_rl_b200.discover import find_attractors_exhaustive
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
    rec["attractor_min_states"] = [m[0] for m in states][:16]
    if profile and kw.get("closure") == "bitset":
        big = max([(len(m), m[0]) for m in states] + list(info.get("oversized", [])))
        rec["largest_closure"] = closure_profile(net, big[1])
    torch.cuda.empty_cache()
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles"))
    ap.add_argument("--wide", action="store_true", help="Bittner-28, bb33 and trap_network(34): r09_reach_wide_probe.json")
    ap.add_argument("--closure", choices=["hash", "bitset"], default="hash",
                    help="bitset: the forward closure over the state bitset, r10_reach_forward_probe.json")
    args = ap.parse_args()
    from helpers import GOLD, make_network, product_net
    from pbn_rl_b200 import PBNNetwork
    pbn28 = product_net("pbn28")
    if args.closure == "bitset":
        from pbn_rl_b200.formats import network_from_bnet
        from reach_forward_oracle import free_block_network
        from test_gpu_reach_wide import trap_network
        net20 = PBNNetwork.from_expressions(*make_network(20, 3, 4, seed=20))
        block = lambda n, free: PBNNetwork.from_expressions(*free_block_network(n, free))
        trap34 = PBNNetwork.from_expressions(*trap_network(34))
        bb33 = network_from_bnet(GOLD / "bb33.bnet")
        big, bits = {"max_attractor_states": 1 << 20}, {"closure": "bitset"}
        runs = [("make_network(20, 3, 4, seed=20)", net20, dict(big), False),
                ("make_network(20, 3, 4, seed=20)", net20, dict(big, **bits), True),
                ("make_network(20, 3, 4, seed=20)", net20, dict(bits), False),
                ("free_block_network(20, 0..17)", block(20, range(18)), dict(bits, max_attractor_states=1 << 18), True),
                ("free_block_network(34, 0..17)", block(34, range(18)), dict(bits, max_attractor_states=1 << 18), True),
                ("free_block_network(34, 0..15 + 32, 33)", block(34, list(range(16)) + [32, 33]),
                 dict(bits, max_attractor_states=1 << 18), True),
                ("free_block_network(34, 0..21)", block(34, range(22)), dict(bits), True)]
        for name, net in (("Bittner-28", pbn28), ("bb33", bb33)):
            runs += [(name, net, {}, False), (name, net, dict(bits), False), (name, net, {}, False),
                     (name, net, dict(bits), True)]
        runs += [("trap_network(34)", trap34, {}, False), ("trap_network(34)", trap34, dict(bits), True)]
        out = {"card": card(), "torch": torch.__version__, "cases": []}
        Path(args.out).mkdir(parents=True, exist_ok=True)
        for name, net, kw, profile in runs:
            out["cases"].append(forward_case(name, net, kw, profile))
            (Path(args.out) / "r10_reach_forward_probe.json").write_text(json.dumps(out, indent=1) + "\n")
        return
    if args.wide:
        from pbn_rl_b200.formats import network_from_bnet
        from test_gpu_reach_wide import trap_network
        runs = [("Bittner-28", pbn28, {}), ("bb33", network_from_bnet(GOLD / "bb33.bnet"), {"partial": False}),
                ("trap_network(34)", PBNNetwork.from_expressions(*trap_network(34)), {"partial": False})]
        fname = "r09_reach_wide_probe.json"
    else:
        net20 = PBNNetwork.from_expressions(*make_network(20, 3, 4, seed=20))
        net24 = PBNNetwork.from_expressions(*make_network(24, 2, 3, seed=24))
        runs = [("Bittner-28", pbn28, {}), ("make_network(20, 3, 4, seed=20)", net20, {}),
                ("make_network(24, 2, 3, seed=24)", net24, {}),
                ("make_network(20, 3, 4, seed=20)", net20, {"max_attractor_states": 1 << 20})]
        fname = "r08_reach_probe.json"
    out = {"card": card(), "torch": torch.__version__, "cases": []}
    Path(args.out).mkdir(parents=True, exist_ok=True)
    for name, net, kw in runs:   # the file is rewritten after every case
        out["cases"].append(case(name, net, **kw))
        (Path(args.out) / fname).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
