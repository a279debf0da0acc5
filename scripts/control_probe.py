"""Device time of the two exact-control operators (pbn_dp_expect, pbn_dp_improve) and of a full "steps" solve.

For each case: CUDA-event time per expect (p = 0 and model A at p = 0.01) and per improve (all genes, 3 flips), the
successor terms sum_u 2^free(u) counted on the device through pbn_successor_sets over all states, terms per second,
improve's coalesced bytes against the HBM bound, and the time of pbn_successor_sets over all states (the predictor
evaluation alone) next to expect's.  Then the wall time of a full "steps" solve of Bittner-10 for every target
(100 stages), and optionally one expect of Bittner-28 at p = 0.  Writes <out>/r06_control_probe.json and
<out>/r06_control_probe_notes.md; the card's name and power limit are read in the same run.

    python scripts/control_probe.py [--out profiles] [--pbn28]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn, min_seconds=0.5, max_reps=200):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    one = a.elapsed_time(b) / 1e3
    reps = int(min(max_reps, max(3, min_seconds / max(one, 1e-6))))
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps, reps


def successor_terms(env):
    n, S = env.n_genes, 1 << env.n_genes
    total, chunk = 0, 1 << 22
    c1 = torch.empty((chunk, 1), dtype=torch.int64, device=env.device)
    c0 = torch.empty_like(c1)
    maxfree = 0
    for s0 in range(0, S, chunk):
        m = min(chunk, S - s0)
        st = torch.arange(s0, s0 + m, dtype=torch.int64, device=env.device).unsqueeze(1)
        rc = env.lib.pbn_successor_sets(env._h, st.data_ptr(), m, c1.data_ptr(), c0.data_ptr(), env._stream())
        assert rc == 0
        fr = (c1[:m, 0] & c0[:m, 0])
        pc = torch.zeros(m, dtype=torch.int64, device=env.device)
        for i in range(n):
            pc += (fr >> i) & 1
        total += int((torch.ones_like(pc) << pc).sum().item())
        maxfree = max(maxfree, int(pc.max().item()))
    return total, maxfree


def successor_sets_time(env):
    S = 1 << env.n_genes
    m = min(S, 1 << 22)
    st = torch.arange(m, dtype=torch.int64, device=env.device).unsqueeze(1)
    c1 = torch.empty((m, 1), dtype=torch.int64, device=env.device)
    c0 = torch.empty_like(c1)

    def run():
        for _ in range(S // m):
            env.lib.pbn_successor_sets(env._h, st.data_ptr(), m, c1.data_ptr(), c0.data_ptr(), env._stream())
    return timed(run)[0]


def improve_bytes(n, genes, kmax):
    """Bytes the improve passes read and write, counted per access (neighbour reads as coalesced streams)."""
    S = 1 << n
    g = bin(genes).count("1")
    total = 0
    for k in range(1, kmax + 1):
        rd = (g + 1) * (8 if k == 1 else 12) + (0 if k == 1 else 12)   # B_{k-1} (w for k = 1) + incumbent v, policy
        wr = 12 + (12 if k < kmax else 0)                                # v, policy (+ B_k)
        total += (rd + wr) * S
    return total


def case(name, net, attrs, out):
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200.control import _Backup
    rec = {"case": name, "n_genes": net.n_genes}
    for mode, p in (("none", 0.0), ("A", 0.01)):
        env = VecPBNEnv(net, 1, attrs, device="cuda:0", perturb_p=p, perturb_mode="A", kernel="scalar")
        bk = _Backup(env)
        u = torch.randn(1 << net.n_genes, dtype=torch.float64, device="cuda:0")
        t, reps = timed(lambda: bk.expect(u))
        rec["expect_s_%s" % mode] = t
        rec["expect_reps_%s" % mode] = reps
        if mode == "none":
            w = bk.expect(u)
            t, reps = timed(lambda: bk.improve(w, (1 << net.n_genes) - 1, 3, -1.0))
            rec["improve_s"] = t
            rec["improve_reps"] = reps
            nb = improve_bytes(net.n_genes, (1 << net.n_genes) - 1, 3)
            rec["improve_bytes"] = nb
            rec["improve_hbm_bound_s"] = nb / HBM_BYTES_PER_S
            rec["improve_over_bound"] = t / (nb / HBM_BYTES_PER_S)
            terms, maxfree = successor_terms(env)
            rec["successor_terms"] = terms
            rec["mean_2pow_free"] = terms / (1 << net.n_genes)
            rec["max_free"] = maxfree
            rec["terms_per_s"] = terms / rec["expect_s_none"]
            rec["successor_sets_s"] = successor_sets_time(env)
        env.close()
        torch.cuda.empty_cache()
    out.append(rec)
    print(json.dumps(rec), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles"))
    ap.add_argument("--pbn28", action="store_true", help="also one expect of Bittner-28 at p = 0")
    args = ap.parse_args()
    from helpers import attractor_set, make_network, product_net
    from pbn_rl_b200 import AttractorSet, PBNNetwork, VecPBNEnv, find_attractors_stg, solve_control
    torch.manual_seed(0)
    res = {"card": card(), "torch": torch.__version__, "cases": []}
    print(res["card"], flush=True)
    case("bittner10", product_net("pbn10"), attractor_set("pbn10"), res["cases"])
    d = json.loads((ROOT / "tests" / "golden" / "control14.json").read_text())
    c14 = PBNNetwork.from_logic_functions(d["genes"], d["logic_functions"])
    case("control14", c14, find_attractors_stg(c14)[0], res["cases"])
    for n, k, a, seed in ((20, 3, 4, 20), (24, 2, 3, 24)):
        genes, exprs = make_network(n, k, a, seed=seed)
        net = PBNNetwork.from_expressions(genes, exprs)
        case("make_network(%d,%d,%d,seed=%d)" % (n, k, a, seed), net, AttractorSet([[tuple([0] * n)]], n), res["cases"])
    # full "steps" solve of Bittner-10, every target, 100 stages
    net, attrs = product_net("pbn10"), attractor_set("pbn10")
    env = VecPBNEnv(net, 1, attrs, device="cuda:0", kernel="scalar")
    solve_control(env, 0, objective="steps")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for t in range(len(attrs)):
        solve_control(env, t, objective="steps")
    torch.cuda.synchronize()
    res["bittner10_steps_solve_all_targets_s"] = time.perf_counter() - t0
    res["bittner10_targets"] = len(attrs)
    env.close()
    if args.pbn28:
        net = product_net("pbn28")
        env = VecPBNEnv(net, 1, attractor_set("pbn28"), device="cuda:0", kernel="scalar")
        from pbn_rl_b200.control import _Backup
        bk = _Backup(env)
        u = torch.randn(1 << 28, dtype=torch.float64, device="cuda:0")
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        w = bk.expect(u)
        b.record()
        torch.cuda.synchronize()
        rec = {"case": "bittner28_expect_p0_single", "expect_s_none": a.elapsed_time(b) / 1e3,
               "launches": int(2 ** 28 / 2 ** 22)}
        terms, maxfree = successor_terms(env)
        rec.update(successor_terms=terms, mean_2pow_free=terms / 2 ** 28, max_free=maxfree,
                   terms_per_s=terms / rec["expect_s_none"], finite=bool(torch.isfinite(w).all().item()))
        res["cases"].append(rec)
        print(json.dumps(rec), flush=True)
        env.close()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "r06_control_probe.json").write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({k: v for k, v in res.items() if k != "cases"}))


if __name__ == "__main__":
    main()
