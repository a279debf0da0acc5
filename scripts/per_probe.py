#!/usr/bin/env python
"""Device times of the prioritised-replay entry points (pbn_per_*) at the in-situ sizes: a push of 2^20 new
transitions into a ring of 2^22, updates of B = 256 / 4096 priorities (1/8 of them duplicated slots) and samples of
B = 256 / 4096.  Each operation is captured R times back to back in a CUDA graph and the replay is timed with CUDA
events, so the figure is device time per call including the gaps between dependent launches but not the Python /
ctypes launch cost.  The trees (5 * 2^22 floats = 80 MB) fit in the 126 MB L2 and stay warm between calls.
Prints one JSON line with the card name and power limit read in the same run."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        out["nvidia_smi"] = q
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = "unavailable: %s" % e
    return out


def time_graph(fn, reps, rounds=5):
    import torch
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    per_call = []
    for _ in range(rounds):
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        per_call.append(e0.elapsed_time(e1) * 1e3 / reps)
    per_call.sort()
    return {"us_median": per_call[len(per_call) // 2], "us_min": per_call[0], "us_max": per_call[-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--capacity", type=int, default=1 << 22)
    ap.add_argument("--push", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=200)
    a = ap.parse_args()
    import ctypes as C

    import torch

    from bench import load_workload
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200._cabi import check
    from pbn_rl_b200.replay import DevicePrioritizedReplay
    dev = torch.device("cuda:0")
    net, attrs = load_workload("pbn28")
    env = VecPBNEnv(net, 1024, attrs, device=dev)
    ring = DevicePrioritizedReplay(env, a.capacity)
    g = torch.Generator(device=dev).manual_seed(0)
    head = [0]

    def push():
        ring.push(head[0], a.push)
        head[0] = (head[0] + a.push) % a.capacity

    for _ in range(a.capacity // a.push):   # fill the ring once
        push()
    ring.size = a.capacity
    res = {"metric": "prioritised replay device time per call (CUDA-graph replay of back-to-back calls)",
           "capacity": a.capacity, "reps": a.reps, "card": card()}
    res["push_%d" % a.push] = time_graph(push, a.reps)
    for b in (256, 4096):
        idx = torch.randint(0, a.capacity, (b,), device=dev, generator=g)
        dup = torch.randint(0, b, (b // 8,), device=dev, generator=g)
        idx[dup] = idx[:1].clone()
        td = torch.randn((b,), device=dev, generator=g)
        res["update_%d" % b] = time_graph(lambda: ring.update_priorities(idx, td), a.reps)
    for b in (256, 4096):
        u = torch.rand((b,), device=dev, generator=g)
        index = torch.empty((b,), dtype=torch.int64, device=dev)
        weight = torch.empty((b,), dtype=torch.float32, device=dev)

        def sample():   # the tree descent alone (DevicePrioritizedReplay.sample adds the pbn_replay_sample gather)
            check(env.lib.pbn_per_sample(env._h, C.byref(ring._p), u.data_ptr(), b, 0.4, index.data_ptr(),
                                         weight.data_ptr(), env._stream()))
        res["sample_%d" % b] = time_graph(sample, a.reps)
        res["sample_gather_%d" % b] = time_graph(lambda: ring.sample(b, beta=0.4, u=u), a.reps)
    total = ring.total()
    res["tree_total"] = total
    res["push_bytes"] = 4 * (2 * a.push * 2)   # leaves + (about as many) internal nodes, sum and min trees
    env.close()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
