#!/usr/bin/env python
"""Cost per update of steady-state recording at 2^20 envs: plain pbn_rollout, pbn_rollout_record with per-gene
marginals only and with marginals + a k = 8 / k = 12 projection, and steady_state_histogram (one pbn_step + projection
ops + one hash insert per update).  Variants alternate within each repeat; every window is at least --window seconds.
Writes one JSON file (default profiles/r05_ssd_probe.json) with the card name and power limit read in the same run."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np
import torch

import bench
from pbn_rl_b200 import VecPBNEnv
from pbn_rl_b200.discover import StateRecorder, steady_state_histogram

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=str(ROOT / "profiles" / "r05_ssd_probe.json"))
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--window", type=float, default=1.0)
ap.add_argument("--envs", type=int, default=1 << 20)
args = ap.parse_args()

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
E = args.envs
GENES = {"pbn28": [0, 3, 7, 11, 14, 18, 21, 27], "pbn70": [0, 5, 12, 31, 40, 63, 64, 69]}
GENES12 = {"pbn28": GENES["pbn28"] + [1, 9, 17, 25], "pbn70": GENES["pbn70"] + [2, 33, 50, 66]}


def timed(fn, n):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn(n)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


rows = []
for name in ("pbn28", "pbn70"):
    net, attrs = bench.load_workload(name)
    for p in (0.0, 1e-3):
        env = VecPBNEnv(net, E, attrs, device="cuda:0", perturb_p=p, perturb_mode="A", horizon=0)
        g = torch.Generator(device="cuda").manual_seed(1)
        for k in range(net.n_words):
            env.state[:, k] = torch.randint(0, 1 << min(net.n_genes - 64 * k, 62), (E,), device="cuda", generator=g)
        env.rollout(256, stats=False)          # into the steady state
        recs = {"marginals": StateRecorder(env, genes=None), "k8": StateRecorder(env, genes=GENES[name]),
                "k12": StateRecorder(env, genes=GENES12[name])}
        variants = {"rollout": lambda n: env.rollout(n, stats=False)}
        for key, rec in recs.items():
            variants["record_" + key] = (lambda r: (lambda n: env.rollout(n, stats=False, recorder=r)))(rec)
        variants["steady_state_histogram_k8"] = lambda n: steady_state_histogram(env, n, genes=GENES[name])
        # size every window to >= args.window seconds from a short calibration run
        steps = {}
        for key, fn in variants.items():
            fn(4)
            n = 16
            while True:
                t = timed(fn, n)
                if t > 0.2 * args.window or n >= 1 << 24:
                    break
                n *= 4
            steps[key] = max(int(n * args.window / t * 1.1), 1)
        times = {key: [] for key in variants}
        for _ in range(args.repeats):
            for key, fn in variants.items():
                times[key].append(timed(fn, steps[key]) / steps[key])
        row = {"net": name, "genes": net.n_genes, "perturb_p": p, "envs": E, "gpu": gpu, "steps_per_window": steps,
               "us_per_update": {k: [1e6 * t for t in v] for k, v in times.items()}}
        base = float(np.mean(times["rollout"]))
        row["mean_us_per_update"] = {k: 1e6 * float(np.mean(v)) for k, v in times.items()}
        row["ratio_to_rollout"] = {k: float(np.mean(v)) / base for k, v in times.items()}
        row["speedup_k8_vs_steady_state_histogram"] = float(np.mean(times["steady_state_histogram_k8"]) / np.mean(times["record_k8"]))
        rows.append(row)
        print(json.dumps({k: row[k] for k in ("net", "perturb_p", "mean_us_per_update", "ratio_to_rollout",
                                               "speedup_k8_vs_steady_state_histogram")}), flush=True)
        env.close()

out = Path(args.out)
out.parent.mkdir(parents=True, exist_ok=True)
out.write_text(json.dumps({"gpu": gpu, "rows": rows}, indent=1))
print("wrote", out)
