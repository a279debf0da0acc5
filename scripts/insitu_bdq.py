#!/usr/bin/env python
"""BASELINE config 5: the train_BDQ.py loop with the GPU env feeding the agent's replay memory, in situ.

The reference's loop (bdq_model/__init__.py:150-237) is: predict -> env.step -> memory.store ->
update_policy, one env instance, python objects in between.  Here the same loop runs over E env
instances with every hand-off on the device:

    obs   = env.observe()                  # pbn_observe: packed state/target -> float [2,E,N]
    q     = net(obs)                       # the agent (library GEMMs; NOT part of the hot path)
    a     = eps-greedy(argmax q)           # uint8 [E,bins]
    ring.step(a)                           # pbn_replay_observe + pbn_step + pbn_replay_commit
    batch = ring.sample(256)               # pbn_replay_sample: gather + unpack to update_policy's tensors
    double-DQN update (bdq_model/__init__.py:100-139)

The agent is a caller of the env, not the product: its network has the layer sizes of
bdq_model/network.py:35-54 (Bilinear(N,N,256) -> 128 -> 64 -> 32, value head, `bins` advantage
heads) written with stock torch modules.  Prints one JSON line with env-steps/s in situ and the
time per phase (CUDA events).

--per: the DDQN+PER variant (ddqn_per/, SURVEY.md section 2 row 13) on the device prioritised replay
(DevicePrioritizedReplay): commit also pushes the new slots into the sum / min trees (timed as `per_push`),
the sample is proportional with importance weights, the loss is mean(w * (expected - cur)^2), and after the
optimiser step the sampled slots get new priorities (timed as `per_update`).  The priority of a transition is
the mean over the action branches of |expected - cur| (one TD error per branch; the mean keeps the scale of a
single-branch agent).  beta is annealed linearly on the host from `beta0` to 1 over the timed iterations.
"""
import argparse
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def build_agent(n_genes, bins, device):
    import torch
    from torch import nn

    class BranchingQ(nn.Module):
        def __init__(self):
            super().__init__()
            self.bilinear = nn.Bilinear(n_genes, n_genes, 256)
            self.trunk = nn.Sequential(nn.LeakyReLU(), nn.Linear(256, 128), nn.LeakyReLU(), nn.Linear(128, 64),
                                       nn.LeakyReLU(), nn.Linear(64, 32), nn.LeakyReLU())
            self.value = nn.Sequential(nn.Linear(32, 64), nn.LeakyReLU(), nn.Linear(64, 1))
            self.adv = nn.ModuleList([nn.Sequential(nn.Linear(32, 64), nn.LeakyReLU(), nn.Linear(64, n_genes + 1))
                                      for _ in range(bins)])

        def forward(self, x):               # x: [2, B, N] (states, targets)
            # Bilinear as one GEMM over the outer product (same function as nn.Bilinear, far less memory traffic)
            b = x.shape[1]
            outer = (x[0].unsqueeze(2) * x[1].unsqueeze(1)).reshape(b, -1)
            h = self.trunk(outer @ self.bilinear.weight.reshape(256, -1).t() + self.bilinear.bias)
            adv = torch.stack([head(h) for head in self.adv], dim=1)
            return self.value(h).unsqueeze(2) + adv - adv.mean(2, keepdim=True)

    return BranchingQ().to(device)


def run(net_name="pbn28", envs=1 << 16, iters=50, warmup=5, batch=256, updates_per_step=1, capacity=None,
        gamma=0.999, lr=1e-4, eps=0.1, device="cuda:0", seed=0, chunk=1 << 18, per=False, alpha=0.6, beta0=0.4):
    import copy

    import torch
    import torch.nn.functional as F

    from bench import ENV_KW, load_workload
    from pbn_rl_b200 import VecPBNEnv
    from pbn_rl_b200.replay import DevicePrioritizedReplay, DeviceReplay

    dev = torch.device(device)
    torch.manual_seed(seed)
    torch.backends.cuda.matmul.allow_tf32 = True   # the agent's GEMMs (0/1 inputs; not the env path)
    net, attrs = load_workload(net_name)
    env = VecPBNEnv(net, envs, attrs, device=dev, auto_reset=True, **ENV_KW)
    env.reset()
    bins, n = env.bins, env.n_genes
    cap = capacity or max(4 * envs, 10_000)
    ring = DevicePrioritizedReplay(env, cap, alpha=alpha) if per else DeviceReplay(env, cap)
    q = build_agent(n, bins, dev)
    target = copy.deepcopy(q)
    adam = torch.optim.Adam(q.parameters(), lr=lr)
    gen = torch.Generator(device=dev).manual_seed(seed)
    obs = torch.empty((2, envs, n), dtype=torch.float32, device=dev)
    greedy = torch.empty((envs, bins), dtype=torch.uint8, device=dev)
    phases = ("observe", "policy", "step+replay", "sample", "update") + (("per_push", "per_update") if per else ())
    ev = {p: [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)] for p in phases}
    acc = dict.fromkeys(phases, 0.0)
    losses, weight_max = [], []
    done_iters = [0]

    def iteration(timed):
        ev["observe"][0].record()
        env.observe(obs)
        ev["observe"][1].record()
        ev["policy"][0].record()
        with torch.no_grad():
            for c0 in range(0, envs, chunk):     # bounds the [B, N*N] outer-product temporary
                greedy[c0:c0 + chunk] = q(obs[:, c0:c0 + chunk]).argmax(dim=2).to(torch.uint8)
            explore = torch.rand((envs, 1), device=dev, generator=gen) < eps
            rnd = torch.randint(0, n + 1, (envs, bins), device=dev, generator=gen, dtype=torch.uint8)
            actions = torch.where(explore, rnd, greedy)
        ev["policy"][1].record()
        ev["step+replay"][0].record()
        if per:   # the uniform ring's three calls, then the tree push timed on its own
            head = ring.head
            ring.observe()
            env.step(actions, final_state=ring._final)
            DeviceReplay.commit(ring, actions, ring._final)
            ev["step+replay"][1].record()
            ev["per_push"][0].record()
            ring.push(head, envs)
            ev["per_push"][1].record()
        else:
            ring.step(actions)
            ev["step+replay"][1].record()
        beta = beta0 + (1.0 - beta0) * min(1.0, done_iters[0] / max(1, iters))
        for _ in range(updates_per_step):
            ev["sample"][0].record()
            b = ring.sample(batch, beta=beta, generator=gen) if per else ring.sample(batch, generator=gen)
            ev["sample"][1].record()
            ev["update"][0].record()
            cur = q(b["obs"]).gather(2, b["actions"]).squeeze(-1)
            with torch.no_grad():
                arg = q(b["next_obs"]).argmax(dim=2)
                nxt = target(b["next_obs"]).gather(2, arg.unsqueeze(2)).squeeze(-1)
                expected = b["reward"] + nxt * gamma * b["done"]   # `masks` = the stored done flag, as the reference
            if per:
                delta = expected - cur
                loss = (b["weight"] * delta * delta).mean()
            else:
                loss = F.mse_loss(expected, cur)
            adam.zero_grad(set_to_none=True)
            loss.backward()
            for p in q.parameters():
                p.grad.clamp_(-1.0, 1.0)
            adam.step()
            ev["update"][1].record()
            if per:
                ev["per_update"][0].record()
                ring.update_priorities(b["index"], delta.detach().abs().mean(dim=1))
                ev["per_update"][1].record()
            if timed:
                losses.append(loss.detach())
                if per:
                    weight_max.append(b["weight"].max())
        if timed:
            torch.cuda.synchronize()
            for p in phases:
                acc[p] += ev[p][0].elapsed_time(ev[p][1])
            done_iters[0] += 1

    for _ in range(warmup):
        iteration(False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        iteration(True)
    e1.record()
    torch.cuda.synchronize()
    secs = max(time.perf_counter() - t0, e0.elapsed_time(e1) * 1e-3)
    stats = env.stats()
    out = {
        "metric": "PBN env-steps/s in situ (BDQ loop, GPU env -> device replay ring -> policy update)",
        "value": envs * iters / secs, "unit": "env-steps/s", "network": net_name, "envs": envs, "iters": iters,
        "batch": batch, "updates_per_step": updates_per_step, "replay_capacity": ring.capacity,
        "replay_bytes_per_transition": ring.bytes_per_transition, "ms_per_iteration": 1e3 * secs / iters,
        "phase_ms_per_iteration": {p: acc[p] / iters for p in phases},
        "loss_last": float(losses[-1].item()) if losses else None, "episodes": stats["episodes"],
        "kernel": env.kernel, "env_launches": env.launches,
    }
    if per:
        out["per"] = {"alpha": alpha, "beta0": beta0, "beta_last": beta0 + (1.0 - beta0) * min(1.0, (iters - 1) / max(1, iters)),
                      "priority": "mean over action branches of |TD error|",
                      "weight_max": max(float(w.item()) for w in weight_max), "total": ring.total(),
                      "pmin": ring.pmin(), "max_p": ring.max_p()}
    env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--net", default="pbn28")
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--updates-per-step", type=int, default=1)
    ap.add_argument("--per", action="store_true", help="prioritised replay (DevicePrioritizedReplay), DDQN+PER loss")
    a = ap.parse_args()
    print(json.dumps(run(a.net, a.envs, a.iters, a.warmup, a.batch, a.updates_per_step, per=a.per)), flush=True)


if __name__ == "__main__":
    main()
