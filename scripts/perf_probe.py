#!/usr/bin/env python
"""Time pbn_step variants on one GPU (CUDA-graph replays, CUDA events).  Development aid."""
import argparse
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import torch  # noqa: E402

import bench  # noqa: E402
from pbn_rl_b200 import VecPBNEnv  # noqa: E402


def time_config(net, attrs, envs, kernel, p, auto_reset, stats, actions, batches=8, graph_steps=32, reps=20, pdl=False, resident=False, chain=False, streams=1):
    dev = torch.device("cuda:0")
    es = []
    for b in range(batches):
        kw = dict(bench.ENV_KW)
        kw["perturb_p"] = p
        e = VecPBNEnv(net, envs, attrs, device=dev, env_offset=b * envs, auto_reset=auto_reset, device_counter=True,
                      kernel=kernel, pdl=pdl, resident=resident, chain=chain, **kw)
        g = torch.Generator(device=dev).manual_seed(b)
        e.state[:, 0] = torch.randint(0, 1 << min(net.n_genes, 62), (envs,), generator=g, device=dev)
        e.set_target(torch.randint(0, len(attrs), (envs,), generator=g, device=dev, dtype=torch.int32))
        es.append(e)
    g = torch.Generator(device=dev).manual_seed(99)
    pool = [torch.randint(0, net.n_genes + 1, (envs, 3), generator=g, device=dev, dtype=torch.uint8) for _ in range(8)]

    def step(i):
        es[i % batches].step(pool[i % 8] if actions else None, stats=stats)

    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for i in range(batches):
            step(i)
        for e in es:
            e.advance_counter()
        s.synchronize()
        # streams > 1: env batch b belongs to stream b % streams; every stream replays its own graph (a PDL sequence over
        # its batches), the graphs of a round are in flight together
        lanes = [s] + [torch.cuda.Stream() for _ in range(streams - 1)]
        graphs = []
        for k, ls in enumerate(lanes):
            gr = torch.cuda.CUDAGraph()
            ls.wait_stream(s)
            with torch.cuda.graph(gr, stream=ls):
                for i in range(graph_steps):
                    if (i % batches) % streams == k:
                        step(i)
                for b, e in enumerate(es):
                    if b % streams == k:
                        e.advance_counter()
            graphs.append(gr)

        def replay_all():
            for ls in lanes[1:]:
                ls.wait_stream(s)
            for gr, ls in zip(graphs, lanes):
                with torch.cuda.stream(ls):
                    gr.replay()
            for ls in lanes[1:]:
                s.wait_stream(ls)

        replay_all()
        s.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        for _ in range(reps):
            replay_all()
        e1.record(s)
        s.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (reps * graph_steps)
    for e in es:
        e.close()
    return us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--net", default="pbn28")
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--kernels", default="sliced")
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--big-attractor", type=int, default=0, help="add one attractor of this many random states (hash-set membership)")
    ap.add_argument("--pdl", action="store_true")
    ap.add_argument("--graph-steps", type=int, default=32)
    ap.add_argument("--streams", type=int, default=1, help="env batches stepped concurrently on this many streams")
    ap.add_argument("--chain", action="store_true", help="tile-level chaining of resident steps (PBN_STEP_CHAIN)")
    ap.add_argument("--batches", type=int, default=8)
    ap.add_argument("--resident", action="store_true", help="plane-resident env state (step_planes.cuh)")
    ap.add_argument("--p", type=float, default=0.001, help="perturbation probability of the 'full' row")
    args = ap.parse_args()
    net, attrs = bench.load_workload(args.net)
    if args.big_attractor:
        import numpy as np
        from pbn_rl_b200 import AttractorSet
        rng = np.random.default_rng(8192)
        big = {tuple(int(v) for v in rng.integers(0, 2, size=net.n_genes)) for _ in range(args.big_attractor + 200)}
        attrs = AttractorSet(list(attrs.attractors) + [sorted(big)[:args.big_attractor]], net.n_genes)
    W = net.n_words
    rows = [("full (p=%g, reset, stats)" % args.p, args.p, True, True, True),
            ("no perturbation", 0.0, True, True, True),
            ("no auto-reset", 0.001, False, True, True),
            ("no stats", 0.001, True, False, True),
            ("no actions", 0.001, True, True, False),
            ("bare (p=0, no reset/stats)", 0.0, False, False, True)]
    if args.quick:
        rows = rows[:1]
    for kernel in args.kernels.split(","):
        for label, p, ar, st, act in rows:
            us = time_config(net, attrs, args.envs, kernel, p, ar, st, act, pdl=args.pdl, graph_steps=args.graph_steps, resident=args.resident or args.chain, chain=args.chain, batches=args.batches)
            gbs = bench.BYTES_PER_STEP[W] * args.envs / us / 1e3
            print(("chain " if args.chain else "resident " if args.resident else "") + "%-8s %-30s %9.2f us/step  %8.3e steps/s  %7.1f GB/s" % (kernel, label, us, args.envs / us * 1e6, gbs), flush=True)


if __name__ == "__main__":
    main()
