#!/usr/bin/env python
"""Batched walk_eval (plen_bullet/src/walk_eval.py:16-104): roll the reference's SHIPPED policy (checkpoint
plen_walk_gazebo_3229999, the one walk_eval.py loads; its actor weights travel in tests/golden/td3_golden.npz) through
the B200 env, deterministic action = actor(state) as in walk_eval.py:79-81.

Besides being the third caller of the env, this is an indirect pin of the physics (SURVEY.md 8c): the policy was trained
against PyBullet's dynamics; if the restated dynamics were far off it would fall at once.  Env 0 is the noise-free
rollout (reset and policy are deterministic, so every noise-free env is identical); the others add N(0, sigma) action
noise to give a distribution.  Reports episode length / return of the first episode and the distance walked.

    python scripts/walk_eval_batched.py [--envs 4096] [--sigma 0.05] [--precision fp32|fp16]
                                        [--mass-scale S] [--payload KG [--payload-offset X Y Z]] [--latency-ticks D | LO:HI]

--mass-scale / --payload sweep the policy's robustness to the robot's mass (PlenVecEnv.set_env_mass): every body x S, and a
point mass of KG kg on the torso, by default at the torso body's centre of mass.  --latency-ticks sweeps its robustness to servo
command latency (PlenVecEnv.set_env_latency): every robot's servos act D physics ticks (4.17 ms each at 240 Hz) late, or a
delay drawn uniformly from LO..HI per robot (seeded).
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from plen_ml_walk_b200.td3 import Actor, actor_forward
from plen_ml_walk_b200.vec_env import PlenVecEnv

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "td3_golden.npz")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--sigma", type=float, default=0.05)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "fp16"])
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--sole-manifold", type=int, default=0, choices=[0, 1],
                    help="plen_config.sole_manifold: 1 = Bullet's one-point-per-tick persistent manifold (profiles/r2_physics_pin.md 5)")
    ap.add_argument("--config", action="append", default=[], metavar="KEY=VALUE",
                    help="plen_config override (repeatable), e.g. --config warmstart_factor=0.85 --config support_tie=0")
    ap.add_argument("--mass-scale", type=float, default=None, help="factor on the mass and inertia of every body")
    ap.add_argument("--payload", type=float, default=None, metavar="KG", help="point mass on the torso, kg")
    ap.add_argument("--payload-offset", type=float, nargs=3, default=None, metavar=("X", "Y", "Z"),
                    help="where the payload sits in the torso body frame, m (default: the torso's centre of mass)")
    ap.add_argument("--latency-ticks", default=None, metavar="D|LO:HI",
                    help="servo command latency in physics ticks (0 .. 2 * substeps), or LO:HI for a uniform draw per robot")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    g = np.load(GOLD)
    actor = Actor().to(dev)
    actor.load_state_dict({k: torch.from_numpy(g["actor_" + k.replace(".", "_")]).to(dev) for k in actor.state_dict().keys()})
    n = a.envs
    ovr = {"sole_manifold": a.sole_manifold}
    for kv in a.config:
        k, v = kv.split("=", 1)
        ovr[k] = float(v) if ("." in v or "e" in v.lower()) else int(v)
    env = PlenVecEnv(n, device=dev, auto_reset=False, config_overrides=ovr)
    mass = None
    if a.mass_scale is not None or a.payload is not None:
        at = list(a.payload_offset) if a.payload_offset is not None else [float(v) for v in env.model.com[0]]
        pay = torch.tensor([a.payload or 0.0] + at, dtype=torch.float32).expand(n, 4)
        env.set_env_mass(None if a.mass_scale is None else torch.full((n,), a.mass_scale), pay if a.payload is not None else None)
        mass = {"mass_scale": a.mass_scale, "payload_kg": a.payload, "payload_at_m": at if a.payload is not None else None}
    latency = None
    if a.latency_ticks is not None:
        lo, _, hi = a.latency_ticks.partition(":")
        lo, hi = int(lo), int(hi or lo)
        gen = torch.Generator(device=dev); gen.manual_seed(0)
        env.set_env_latency(torch.randint(lo, hi + 1, (n,), device=dev, generator=gen))
        latency = {"ticks_lo": lo, "ticks_hi": hi, "ms_per_tick": 1000.0 * float(env.cfg.dt)}
    state = env.reset().clone()
    alive = torch.ones(n, dtype=torch.bool, device=dev)
    ep_len = torch.zeros(n, device=dev); ep_ret = torch.zeros(n, device=dev)
    x_end = torch.zeros(n, device=dev)
    for t in range(a.steps):
        act = actor_forward(actor, state, noise_std=a.sigma, seed=t + 1, precision=a.precision)
        clean = actor_forward(actor, state[:1], precision=a.precision)
        act[0] = clean[0]                                                    # env 0: the deterministic walk_eval rollout
        obs, r, done, info = env.step(act)
        ep_len += alive
        ep_ret += torch.where(alive, r, torch.zeros_like(r))
        qpos = env.get_state()[0]
        x_end = torch.where(alive, qpos[:, 0], x_end)
        alive &= ~done
        state = obs.clone()
    L, R, X = ep_len.cpu().numpy(), ep_ret.cpu().numpy(), x_end.cpu().numpy()
    print(json.dumps({
        "policy": "plen_walk_gazebo_3229999 (reference checkpoint)", "envs": n, "steps": a.steps, "sigma": a.sigma,
        "precision": a.precision, "sole_manifold": a.sole_manifold, "config_overrides": ovr, "mass": mass, "latency": latency,
        "deterministic": {"episode_length": float(L[0]), "return": float(R[0]), "x_final_m": float(X[0])},
        "noisy": {"episode_length_mean": float(L[1:].mean()), "episode_length_median": float(np.median(L[1:])),
                  "survived_all_steps_frac": float((L[1:] >= a.steps).mean()), "return_mean": float(R[1:].mean()),
                  "return_quantiles_5_25_50_75_95": [float(q) for q in np.quantile(R[1:], [0.05, 0.25, 0.5, 0.75, 0.95])],
                  "x_final_mean_m": float(X[1:].mean()), "x_final_std_m": float(X[1:].std())}}))


if __name__ == "__main__":
    main()
