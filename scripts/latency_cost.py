#!/usr/bin/env python
"""Cost of per-robot servo command latency in plen_step: two arms timed in one process, alternating pass by pass.

    python scripts/latency_cost.py [--sizes 131072 1048576] [--passes 5] [--steps 20] [--warmup 5]

  stock    a context that never called set_env_latency (no command history: k_dyn reads the targets as before)
  latency  set_env_latency with a delay drawn uniformly from 0..2 * substeps ticks per robot: every tick of k_dyn reads at most
           one 128-byte history row per robot, and tick 0 also writes one

Each pass times `--steps` random-action env steps (auto-reset on) with CUDA events after `--warmup` untimed ones; the arms take
turns, so drifts of the clock or of other work on the machine hit both alike.  Prints ms per step (median and min..max over
the passes) and the latency arm's median relative to stock, with the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from plen_ml_walk_b200.vec_env import PlenVecEnv


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (x.strip() for x in out.split(",", 1))
        return name, power
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def make_arm(kind, n, dev, seed):
    env = PlenVecEnv(n, device=dev)
    if kind == "latency":
        g = torch.Generator(device=dev); g.manual_seed(seed)
        env.set_env_latency(torch.randint(0, env.max_latency_ticks + 1, (n,), device=dev, generator=g))
    env.reset()
    return env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[131072, 1048576])
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    name, power = card()
    arms = ("stock", "latency")
    result = {"card": name, "power_limit": power, "passes": a.passes, "steps": a.steps, "sizes": {}}
    for n in a.sizes:
        envs = {k: make_arm(k, n, dev, seed=i + 1) for i, k in enumerate(arms)}
        g = torch.Generator(device=dev); g.manual_seed(0)
        acts = [torch.empty((n, 18), device=dev).uniform_(-1, 1, generator=g) for _ in range(8)]
        ms = {k: [] for k in arms}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for p in range(a.passes):
            for k in (arms if p % 2 == 0 else arms[::-1]):
                env = envs[k]
                for w in range(a.warmup):
                    env.step(acts[w % 8])
                torch.cuda.synchronize()
                e0.record()
                for s in range(a.steps):
                    env.step(acts[s % 8])
                e1.record()
                torch.cuda.synchronize()
                ms[k].append(e0.elapsed_time(e1) / a.steps)
        faults = {k: envs[k].fault_count() for k in arms}
        del envs
        torch.cuda.empty_cache()
        row = {}
        for k in arms:
            v = np.array(ms[k])
            row[k] = {"ms_per_step_median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()),
                      "spread_pct": float(100 * (v.max() - v.min()) / np.median(v)),
                      "vs_stock_pct": float(100 * (np.median(v) / np.median(ms["stock"]) - 1)), "faults": faults[k]}
            print("%9d robots  %-7s  %.3f ms/step  (%.3f .. %.3f, spread %.1f %%)  %+.2f %% vs stock  [%s, %s]"
                  % (n, k, row[k]["ms_per_step_median"], v.min(), v.max(), row[k]["spread_pct"], row[k]["vs_stock_pct"], name, power))
        result["sizes"][str(n)] = row
    print(json.dumps(result))


if __name__ == "__main__":
    main()
