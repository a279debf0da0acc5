"""PCIe copy rates and pbn_step_host timing for several lane counts, every result form (tuning aid, not a bench).
Lane count 0 is the library default."""
import sys, time
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch
from bench import load_workload, ENV_KW
from pbn_rl_b200 import VecPBNEnv

def timeit(fn, n=20):
    for _ in range(3): fn()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(n): fn()
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / n

dev = torch.device("cuda:0")
for mb in (1, 4, 16, 64):
    n = mb << 20
    h = torch.empty(n, dtype=torch.uint8, pin_memory=True); d = torch.empty(n, dtype=torch.uint8, device=dev)
    t1 = timeit(lambda: d.copy_(h, non_blocking=True)); t2 = timeit(lambda: h.copy_(d, non_blocking=True))
    print("copy %3d MB: H2D %.1f GB/s  D2H %.1f GB/s" % (mb, n / t1 / 1e9, n / t2 / 1e9))
net, attrs = load_workload("pbn28")
E = 1 << 20
env = VecPBNEnv(net, E, attrs, device=dev, auto_reset=True, **ENV_KW)
env.reset()
pa = env.pinned_actions(); pa.random_(0, 29)
import numpy as np
a16 = env.pinned_actions16(); a16.numpy().view(np.uint16)[...] = env.pack_actions16(pa.numpy())
for compact in (False, True, "packed"):
    for ch in (0, 1, 2, 3, 4, 6, 8):
        if compact == "packed":
            t = timeit(lambda: env.step_host(None, chunks=ch, compact="packed", actions16=a16))
        else:
            t = timeit(lambda: env.step_host(pa, chunks=ch, compact=compact))
        print("step_host compact=%s lanes=%2d: %.3f ms  %.3e env-steps/s" % (compact, ch, t * 1e3, E / t))
