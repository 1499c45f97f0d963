#!/usr/bin/env python
"""Cost of per-robot observation noise in plen_step: two arms timed in one process, alternating pass by pass.

    python scripts/obs_noise_cost.py [--sizes 131072 1048576] [--passes 5] [--steps 20] [--warmup 5]

  stock  a context that never called set_obs_noise (k_post's stock instance)
  noise  set_obs_noise with white noise on every continuous word, a per-episode bias on every word and contact flips at
         p = 0.05: k_post's noise instance reads one 384-byte noise row per robot, draws 24 Gaussians and two flips per step
         (three Gaussians per word more for a robot that auto-resets) and writes the clean observation next to the noisy one

Each pass times `--steps` random-action env steps (auto-reset on) with CUDA events after `--warmup` untimed ones; the arms take
turns, so drifts of the clock or of other work on the machine hit both alike.  Prints ms per step (median and min..max over
the passes) and the noise arm's median relative to stock, with the card's name and power limit.
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


def make_arm(kind, n, dev):
    env = PlenVecEnv(n, device=dev)
    if kind == "noise":
        env.set_obs_noise(std=0.01, bias_std=0.02, contact_flip=0.05, seed=1)
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
    arms = ("stock", "noise")
    result = {"card": name, "power_limit": power, "passes": a.passes, "steps": a.steps, "sizes": {}}
    for n in a.sizes:
        envs = {k: make_arm(k, n, dev) for k in arms}
        g = torch.Generator(device=dev); g.manual_seed(0)
        acts = [torch.empty((n, 18), device=dev).uniform_(-1, 1, generator=g) for _ in range(8)]
        ms = {k: [] for k in arms}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for p in range(a.passes):
            for k in (arms if p % 2 == 0 else arms[::-1]):
                env = envs[k]
                for w in range(a.warmup):
                    env.lib.plen_step(env._ctx, env._p(acts[w % 8]), env._p(env._obs), env._p(env._reward), env._p(env._done),
                                      env._p(env._timeout), env._p(env._terminal_obs), env._stream())
                torch.cuda.synchronize()
                e0.record()
                for s in range(a.steps):
                    env.lib.plen_step(env._ctx, env._p(acts[s % 8]), env._p(env._obs), env._p(env._reward), env._p(env._done),
                                      env._p(env._timeout), env._p(env._terminal_obs), env._stream())
                e1.record()
                torch.cuda.synchronize()
                ms[k].append(e0.elapsed_time(e1) / a.steps)
        del envs
        torch.cuda.empty_cache()
        row = {}
        for k in arms:
            v = np.array(ms[k])
            row[k] = {"ms_per_step_median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()),
                      "spread_pct": float(100 * (v.max() - v.min()) / np.median(v)),
                      "vs_stock_pct": float(100 * (np.median(v) / np.median(ms["stock"]) - 1))}
            print("%9d robots  %-5s  %.3f ms/step  (%.3f .. %.3f, spread %.1f %%)  %+.2f %% vs stock  [%s, %s]"
                  % (n, k, row[k]["ms_per_step_median"], v.min(), v.max(), row[k]["spread_pct"], row[k]["vs_stock_pct"], name, power))
        result["sizes"][str(n)] = row
    print(json.dumps(result))


if __name__ == "__main__":
    main()
