#!/usr/bin/env python
"""Cost of per-robot reset states (PlenVecEnv.settle_resets): the settle itself, and plen_step with a reset table.

    python scripts/reset_cost.py [--settle-sizes 4096 131072 1048576] [--step-sizes 131072 1048576] [--passes 5] [--steps 20]
                                 [--warmup 5]

  settle   settle_resets() of every robot from random start poses under random scales and masses (reset_ticks physics ticks over
           the whole batch plus two small kernels), timed with CUDA events, one call per pass after one untimed call, alternating
           with one env step of the same context (substeps ticks plus k_post) timed the same way
  step     `--steps` random-action env steps (auto-reset on) after `--warmup` untimed ones, two arms alternating pass by pass:
           stock (no reset table) and settled (a table settled from random headings, so that every reset restores a per-robot
           row instead of the shared snapshot)

Prints ms (median and min..max over the passes) with the card's name and power limit, then one JSON line.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from mass_dr_cost import card
from plen_ml_walk_b200.vec_env import PlenVecEnv


def rand_params(env, n, dev, seed):
    g = torch.Generator(device=dev); g.manual_seed(seed)
    u = lambda shape, lo, hi: torch.empty(shape, device=dev).uniform_(lo, hi, generator=g)
    env.set_env_scales(friction=u(n, 0.6, 1.2), motor_force=u(n, 0.8, 1.2), motor_gain=u(n, 0.8, 1.1))
    pay = torch.cat([u((n, 1), 0.0, 0.1), torch.tensor([float(v) for v in env.model.com[0]], device=dev) + u((n, 3), -0.01, 0.01)], 1)
    env.set_env_mass(u((n, 19), 0.8, 1.2), pay)
    pose = torch.stack([u(n, -1, 1), u(n, -1, 1), torch.full((n,), 0.158, device=dev), u(n, -3.14, 3.14)], 1)
    return pose


def stats(v, ref=None):
    v = np.array(v)
    d = {"ms_median": float(np.median(v)), "min": float(v.min()), "max": float(v.max())}
    if ref is not None:
        d["vs_stock_pct"] = float(100 * (np.median(v) / np.median(ref) - 1))
    return d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--settle-sizes", type=int, nargs="+", default=[4096, 131072, 1048576])
    ap.add_argument("--step-sizes", type=int, nargs="+", default=[131072, 1048576])
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    name, power = card()
    result = {"card": name, "power_limit": power, "passes": a.passes, "steps": a.steps, "settle": {}, "step": {}}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g = torch.Generator(device=dev); g.manual_seed(0)
    for n in a.settle_sizes:
        env = PlenVecEnv(n, device=dev)
        pose = rand_params(env, n, dev, seed=1)
        act = torch.empty((n, 18), device=dev).uniform_(-1, 1, generator=g)
        env.reset()
        env.settle_resets(start_pose=pose)
        env.step(act)
        settle, step = [], []
        for p in range(a.passes):
            for kind in (("settle", "step") if p % 2 == 0 else ("step", "settle")):
                torch.cuda.synchronize()
                e0.record()
                if kind == "settle":      # the library call alone (settle_resets also validates the poses on the host)
                    assert env.lib.plen_settle_env_resets(env._ctx, env._p(pose), env._stream()) == 0
                else:
                    env.step(act)
                e1.record()
                torch.cuda.synchronize()
                (settle if kind == "settle" else step).append(e0.elapsed_time(e1))
        row = {"settle": stats(settle), "one_step": stats(step), "settle_over_step": float(np.median(settle) / np.median(step))}
        result["settle"][str(n)] = row
        print("%9d robots  settle_resets %.3f ms (%.3f .. %.3f)  one env step %.3f ms  ratio %.2f  [%s, %s]"
              % (n, row["settle"]["ms_median"], row["settle"]["min"], row["settle"]["max"], row["one_step"]["ms_median"],
                 row["settle_over_step"], name, power))
        del env
        torch.cuda.empty_cache()
    for n in a.step_sizes:
        envs = {"stock": PlenVecEnv(n, device=dev), "settled": PlenVecEnv(n, device=dev)}
        gg = torch.Generator(device=dev); gg.manual_seed(2)
        yaw = torch.empty(n, device=dev).uniform_(-3.14, 3.14, generator=gg)
        envs["settled"].settle_resets(start_pose=torch.stack([torch.zeros(n, device=dev), torch.zeros(n, device=dev),
                                                              torch.full((n,), 0.158, device=dev), yaw], 1))
        for env in envs.values():
            env.reset()
        acts = [torch.empty((n, 18), device=dev).uniform_(-1, 1, generator=g) for _ in range(8)]
        ms = {k: [] for k in envs}
        for p in range(a.passes):
            for k in (("stock", "settled") if p % 2 == 0 else ("settled", "stock")):
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
        row = {k: stats(ms[k], ms["stock"]) for k in envs}
        result["step"][str(n)] = row
        for k in envs:
            print("%9d robots  %-7s  %.3f ms/step  (%.3f .. %.3f)  %+.2f %% vs stock  [%s, %s]"
                  % (n, k, row[k]["ms_median"], row[k]["min"], row[k]["max"], row[k]["vs_stock_pct"], name, power))
        del envs
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
