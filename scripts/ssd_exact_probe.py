"""Device time of the exact forward operator pbn_dp_push against pbn_dp_expect, and of the stationary solver.

1. On the networks of control_probe.py (Bittner-10, control14, make_network(20, 3, 4, seed=20),
   make_network(24, 2, 3, seed=24)), at p = 0 and model A at p = 0.01: CUDA-event time per push (a random
   distribution with every entry > 0, so every state's terms run) and per expect, successor terms per second of each.
2. One point-mass push on Bittner-28 (the state with the most free genes among 2^16 random ones).
3. Iterations and wall time of stationary_distribution(tol = 1e-10) on make_network(20, 3, 4, seed=20) at model A
   p = 1e-2 and 1e-3.
Writes <out>/r07_ssd_exact_probe.json; the card's name and power limit are read in the same run.

    python scripts/ssd_exact_probe.py [--out profiles]
"""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "tests"), str(ROOT / "scripts")]

from control_probe import card, successor_terms, timed  # noqa: E402


def case(name, net, attrs):
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200.control import _Backup
    S = 1 << net.n_genes
    rec = {"case": name, "n_genes": net.n_genes}
    for mode, p in (("none", 0.0), ("A", 0.01)):
        env = VecPBNEnv(net, 1, attrs, device="cuda:0", perturb_p=p, perturb_mode="A", kernel="scalar")
        bk = _Backup(env)
        u = torch.randn(S, dtype=torch.float64, device="cuda:0")
        x = torch.rand(S, dtype=torch.float64, device="cuda:0") + 0.5
        x /= x.sum()
        rec["expect_s_%s" % mode] = timed(lambda: bk.expect(u))[0]
        rec["push_s_%s" % mode], rec["push_reps_%s" % mode] = timed(lambda: bk.push(x))
        rec["push_over_expect_%s" % mode] = rec["push_s_%s" % mode] / rec["expect_s_%s" % mode]
        if mode == "none":
            terms, maxfree = successor_terms(env)
            rec.update(successor_terms=terms, max_free=maxfree)
        rec["push_terms_per_s_%s" % mode] = rec["successor_terms"] / rec["push_s_%s" % mode]
        rec["expect_terms_per_s_%s" % mode] = rec["successor_terms"] / rec["expect_s_%s" % mode]
        env.close()
        del bk, u, x
        torch.cuda.empty_cache()
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles"))
    args = ap.parse_args()
    import control_oracle as CO
    from helpers import attractor_set, make_network, product_net
    from pbn_rl_b200 import AttractorSet, PBNNetwork, VecPBNEnv, find_attractors_stg, stationary_distribution
    from pbn_rl_b200.control import _Backup
    torch.manual_seed(0)
    res = {"card": card(), "torch": torch.__version__, "cases": []}
    print(res["card"], flush=True)
    res["cases"].append(case("bittner10", product_net("pbn10"), attractor_set("pbn10")))
    d = json.loads((ROOT / "tests" / "golden" / "control14.json").read_text())
    c14 = PBNNetwork.from_logic_functions(d["genes"], d["logic_functions"])
    res["cases"].append(case("control14", c14, find_attractors_stg(c14)[0]))
    net20 = None
    for n, k, a, seed in ((20, 3, 4, 20), (24, 2, 3, 24)):
        net = PBNNetwork.from_expressions(*make_network(n, k, a, seed=seed))
        net20 = net if n == 20 else net20
        res["cases"].append(case("make_network(%d,%d,%d,seed=%d)" % (n, k, a, seed), net,
                                 AttractorSet([[tuple([0] * n)]], n)))
    # one point-mass push on Bittner-28
    net = product_net("pbn28")
    cand = np.random.default_rng(28).integers(0, 1 << 28, size=1 << 16)
    free = CO.free_counts(net, cand)
    s = int(cand[int(free.argmax())])
    env = VecPBNEnv(net, 1, attractor_set("pbn28"), device="cuda:0", kernel="scalar")
    bk = _Backup(env)
    e = torch.zeros(1 << 28, dtype=torch.float64, device="cuda:0")
    e[s] = 1.0
    t, reps = timed(lambda: bk.push(e), max_reps=20)
    rec = {"case": "bittner28_point_mass_push", "state": s, "free": int(free.max()), "terms": 1 << int(free.max()),
           "push_s": t, "reps": reps, "hbm_bytes_min": 4 * 8 << 28,
           "note": "one pass over x, a memset and the fp64 conversion of y: 4 x 8 B per state at least"}
    res["cases"].append(rec)
    print(json.dumps(rec), flush=True)
    env.close()
    del bk, e
    torch.cuda.empty_cache()
    # stationary solves on the 20-gene network
    res["stationary"] = []
    for p in (1e-2, 1e-3):
        env = VecPBNEnv(net20, 1, AttractorSet([[tuple([0] * 20)]], 20), device="cuda:0", perturb_p=p,
                        perturb_mode="A", kernel="scalar")
        stationary_distribution(env, max_iters=16)        # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dist = stationary_distribution(env, tol=1e-10)
        torch.cuda.synchronize()
        rec = {"case": "make_network(20,3,4,seed=20) model A p=%g" % p, "tol": 1e-10, "iterations": dist.iterations,
               "residual": dist.residual, "converged": dist.converged, "wall_s": time.perf_counter() - t0}
        res["stationary"].append(rec)
        print(json.dumps(rec), flush=True)
        env.close()
    big = [c for c in res["cases"] if c.get("n_genes") in (20, 24)]
    res["goals"] = {
        "push_within_2x_of_expect_20_24": all(c["push_over_expect_%s" % m] <= 2.0 for c in big for m in ("none", "A")),
        "stationary_20_p1e-2_under_60s": res["stationary"][0]["converged"] and res["stationary"][0]["wall_s"] < 60.0,
    }
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "r07_ssd_exact_probe.json").write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res["goals"]))


if __name__ == "__main__":
    main()
