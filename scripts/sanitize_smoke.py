"""One small invocation of every kernel of libpbn_b200.so (for compute-sanitizer memcheck / racecheck runs):
both step kernels on ragged batches, reset, auto-reset, host path (zero-copy + copy engine), replay ring,
observation, evaluator bookkeeping, visit-count hash, closure search, wide predictors."""
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import numpy as np
import torch

from helpers import GOLD, attractor_set, product_net
from pbn_rl_b200 import PBNNetwork, VecPBNEnv
from pbn_rl_b200.discover import StateRecorder, VisitCounter, find_attractors_rollout, steady_state_histogram
from pbn_rl_b200.evaluate import evaluate_all_pairs, hamming_policy
from pbn_rl_b200.replay import DeviceReplay

rng = np.random.default_rng(0)
for name, e in (("pbn28", 1024 + 77), ("pbn70", 1500), ("pbn7", 33)):
    net, attrs = product_net(name), attractor_set(name)
    for kernel in ("auto", "scalar"):
        env = VecPBNEnv(net, e, attrs, device="cuda:0", perturb_p=0.05, auto_reset=True, kernel=kernel, horizon=4)
        env.reset()
        ring = DeviceReplay(env, 2 * e + 5)
        for step in range(5):
            act = torch.from_numpy(rng.integers(0, net.n_genes + 1, size=(e, 3), dtype=np.uint8)).cuda()
            ring.step(act)
        ring.sample(64)
        env.observe()
        env.unpack(dtype=torch.float32)
        env.attractor_ids()
        env.step_host(act.cpu().numpy(), chunks=2)
        if net.n_genes <= 32:
            env.step_host(None, compact=True)
        sel = torch.zeros((e, net.n_genes), dtype=torch.uint8)
        env.step_injected(act, sel, torch.zeros((e, net.n_words), dtype=torch.int64))
        table = VisitCounter(env, 1 << 12)
        table.add()
        table.items()
        torch.cuda.synchronize()
        env.close()
m, data = evaluate_all_pairs(product_net("pbn7"), attractor_set("pbn7"), hamming_policy(3), runs=2, max_steps=10)
found, info = find_attractors_rollout(product_net("pbn10"), n_rollouts=2048, burn_in=50)
want = json.loads((GOLD / "control14.json").read_text())
wide = PBNNetwork.from_logic_functions(want["genes"], want["logic_functions"])
env = VecPBNEnv(wide, 777, None, device="cuda:0", perturb_p=0.01)
env.state.random_(0, 1 << 14)
for _ in range(3):
    env.step(None)
steady_state_histogram(env, steps=3)
torch.cuda.synchronize()
env.close()
# round 2: plane-resident kernels (PDL + tile-chained), the general row kernel with the hash set and single-state
# targets in shared memory, genes with up to 8 predictors (third selection plane), packed host path (lanes + graph replay)
from pbn_rl_b200 import AttractorSet
net, attrs = product_net("pbn28"), attractor_set("pbn28")
for chain in (False, True):
    env = VecPBNEnv(net, 2048 + 5, attrs, device="cuda:0", perturb_p=0.05, auto_reset=True, horizon=4, resident=True, chain=chain)
    env.reset()
    for step in range(4):
        env.step(torch.from_numpy(rng.integers(0, 29, size=(2053, 3), dtype=np.uint8)).cuda())
    env.advance_counter()
    env.state.sum().item()
    env.close()
big = sorted({tuple(int(v) for v in rng.integers(0, 2, size=28)) for _ in range(400)})[:300]
env = VecPBNEnv(net, 3000, AttractorSet(list(attrs.attractors) + [big], 28), device="cuda:0", perturb_p=0.05, auto_reset=True, horizon=4)
env.reset()
for step in range(4):
    env.step(torch.from_numpy(rng.integers(0, 29, size=(3000, 3), dtype=np.uint8)).cuda())
env.close()
genes = ["m%d" % i for i in range(9)]
many = PBNNetwork.from_expressions(genes, [["m1", "m2", "m3", "m4", "m5"], [("m0", 0.1), ("m2", 0.2), ("m3", 0.3), ("m4", 0.1), ("m5", 0.1), ("m6 & m7", 0.2)],
                                           ["m0 | m1", "m3", "m4", "m5", "m6", "m7", "~m8"], [("m%d" % j, 0.125) for j in range(8)],
                                           ["m0", "m1", "m2"], ["m8"], ["m1"], ["m2", "m3 | m4"], ["m0"]])
env = VecPBNEnv(many, 1500, None, device="cuda:0", perturb_p=0.02)
assert env.kernel == "sliced"
for _ in range(3):
    env.step(torch.from_numpy(rng.integers(0, 10, size=(1500, 3), dtype=np.uint8)).cuda())
env.rollout(5)
rec = StateRecorder(env, genes=[8, 0, 5])     # pbn_rollout_record (ragged last tile) and pbn_record_states
env.rollout(5, recorder=rec, stride=2)
rec.add()
env.close()
if "--host-lanes" in sys.argv:   # 2^18 envs: slow under the sanitizer's racecheck
    e = 1 << 18
    env = VecPBNEnv(net, e, attrs, device="cuda:0", perturb_p=0.001, auto_reset=True, horizon=20, device_counter=True)
    env.reset()
    a16 = env.pinned_actions16()
    a16.numpy().view(np.uint16)[...] = env.pack_actions16(rng.integers(0, 29, size=(e, 3), dtype=np.uint8))
    for _ in range(4):
        env.step_host(None, compact="packed", actions16=a16)
    env.close()
torch.cuda.synchronize()
print("sanitize_smoke ok:", len(found), "attractors,", int(m.sum()), "evaluator steps")
