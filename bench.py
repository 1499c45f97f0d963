#!/usr/bin/env python
"""bench.py -- PLEN env-steps/sec on B200 (BASELINE.json metric) with roofline, end-to-end and CPU-baseline legs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--total-envs T | --envs-per-gpu E] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one vectorised env step (1 action -> 4 physics ticks -> obs/reward/done/auto-reset) of every env of the
rank: 3 launches per tick (k_dyn, k_rank, k_solve) + k_post (+ the rare-path k_solve_x).  Workload = BASELINE config 5
AS WRITTEN: T = 1,048,576 envs in total, split evenly over the N GPUs of the run (all of them on ONE GPU at N = 1:
7.1 GB of the 180 GB), actions U(-1,1)^18 drawn on the device with torch.Generator(seed 0 + rank), auto-reset on.  The
total is fixed, so the 1 -> 8 GPU curve is STRONG scaling ("scaling": "strong"); `--envs-per-gpu E` fixes the per-GPU
size instead (weak scaling; 131,072 is round 1's shard and is reported under other_configs at N = 1).  Envs are
independent, so ranks share nothing on the data path; torch.distributed (NCCL) is used only for the barrier and the
max-over-ranks of the device time.

`--impl reference` times the reference's CPU implementation of the path on the host cores: the reference's own
PlenWalkEnv on PyBullet (one process per core, kind "pybullet") when `pybullet` is importable (also probed under
baseline/_ref) and the reference checkout is present; otherwise -- as in this image, where neither exists (SURVEY.md
section 8c) -- the float64 oracle PORT (oracle/plen_oracle.c, one thread per core), labelled as such and never
presented as a PyBullet number.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "PLEN env-steps/sec"
UNIT = "env-steps/s"
# algorithmic HBM bytes per env-step (DESIGN.md "Data layout"): state record 96 words read + written, action 18 f32,
# obs 26 f32, reward f32, done + timeout bytes
BYTES_PER_ENV_STEP = 2 * 96 * 4 + 18 * 4 + 26 * 4 + 4 + 2
TICKS_PER_STEP = 4
# measured DRAM traffic of one k_solve launch per robot (ncu --set full, profiles/r1_v9_summary.md): it reads the
# 6.4 KB solve record k_dyn wrote for the tick -- a deliberate trade of HBM bytes for issue slots (DESIGN.md)
SOLVE_DRAM_BYTES_PER_ROBOT = (207.10e6 + 9.92e6) / 32768
# FROZEN in BASELINE.md ("Work per env-step"): executed FP32 work per robot-tick ON THIS WORKLOAD, counted from the SASS-level
# execution counts of ncu's source page (scripts/flops_sass.py: FFMA2 = 4 flop, FFMA = 2, FADD / FMUL = 1 per predicated-on
# thread instruction) over every launch of ONE env step of 131,072 robots at step 30 after the reset, the middle of the
# timed region (profiles/r2_flops_sass.md, final build): k_dyn 44.0 kflop, k_solve 163.9 kflop + k_solve_x 12.0 kflop (the
# bracket of "k_solve" covers both), k_post 17.0 kflop per env step.  The earlier figure (25.9 + 2.7 kflop for the solve) came from
# smsp__sass_thread_inst_executed_op_{fadd,fmul,ffma}_pred_on, which do NOT count the packed FFMA2 (fma.rn.f32x2) that
# carries every row update of k_solve: 28.9 % of its issued instructions, 82 % of its flops (cross-checked against
# sm__pipe_fma_cycles_active of the same launches to 1.9 %).
FLOP_DYN_PER_ROBOT_TICK, FLOP_SOLVE_PER_ROBOT_TICK, FLOP_POST_PER_ENV_STEP = 44.0e3, 175.9e3, 17.0e3
# what ncu's three op metrics see of the same step (scalar FADD + FMUL + 2 FFMA only): kept for comparison with round 1 / 2 lines
FLOP_PER_ENV_STEP_NCU_OP_METRICS = 0.323e6
FLOP_PER_ENV_STEP = 4 * (FLOP_DYN_PER_ROBOT_TICK + FLOP_SOLVE_PER_ROBOT_TICK) + FLOP_POST_PER_ENV_STEP
# the same workload through the REFERENCE ALGORITHM (33-link ABA + velocity-space PGS with 24-wide rows), counted by the
# oracle's instrumented FLOP counter (plen_oracle_state.flops; scripts/oracle_flops.py): 1.32 Mflop per env-step
REF_ALGO_FLOP_PER_ENV_STEP = 1.32e6
FP32_NOMINAL_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12          # SURVEY.md section 8d
# --dump-outputs: a step hands its caller 55 floats per env (obs 26, reward, done, timeout, terminal_obs 26), 220 bytes in
# float32; at most this many envs are written (57.7 MB), a fixed seeded sample of them when the run has more
DUMP_MAX_ENVS = 262144


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def wait_first(self, timeout=4.0):
        """nvidia-smi takes a while to print its first line (longer on an 8-GPU box): block until it does."""
        t0 = time.time()
        while self.proc and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.02)

    def count_in(self, t0, t1):
        return sum(1 for ts, _ in self.rows if t0 <= ts <= t1)

    def stop(self, t0=None, t1=None):
        """Median SM clock / throttle reasons of the samples taken in [t0, t1] (all samples when no window is given)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for ts, r in self.rows if t0 is None or t0 <= ts <= t1]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for k, nme in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_port_throughput(n_threads, envs_per_thread, steps, seed=0):
    """env-steps/s of the float64 oracle (kind "port") on n_threads host threads, random actions, auto-reset."""
    from oracle.oracle import PlenOracle
    n = n_threads * envs_per_thread
    o = PlenOracle(n, n_threads=n_threads)
    o.reset()
    rng = np.random.default_rng(seed)
    acts = rng.uniform(-1, 1, (steps + 1, n, 18))
    o.step(acts[0], auto_reset=True)
    t0 = time.perf_counter()
    for s in range(steps):
        o.step(acts[s + 1], auto_reset=True)
    dt = time.perf_counter() - t0
    return n * steps / dt, dt, n


def pybullet_throughput(steps, n_procs):
    """env-steps/s of the reference's own PlenWalkEnv on PyBullet DIRECT, one process per host core (kind "pybullet");
    None when PyBullet or the reference checkout is not reachable (the case in this image)."""
    from oracle import pybullet_ref
    if not pybullet_ref.available():
        return None
    return pybullet_ref.timed_throughput(steps, n_procs)


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    pb = None
    try:
        pb = pybullet_throughput(max(200, 20 * args.steps), cores)
    except Exception as e:                                # a broken PyBullet install must not take the arm down
        sys.stderr.write("pybullet arm failed (%s); falling back to the oracle port\n" % e)
    if pb is not None:
        val, dt, n, kind = pb["value"], pb["seconds"], pb["envs"], "pybullet"
        sample = "%d processes x 1 env x %d steps of the reference's PlenWalkEnv (PyBullet %s, DIRECT)" % (n, pb["steps"], pb["version"])
    else:
        # one "step" = one vector step of cores*E envs on all host threads; E sized from a probe so a step is ~0.3 s and
        # the whole --steps K run stays within a few minutes
        probe, _, _ = cpu_port_throughput(cores, 8, 4, seed=1)
        per_step = min(0.3, 150.0 / max(1, args.steps))
        envs_per_thread = int(max(8, min(4096, probe * per_step / cores)))
        val, dt, n = cpu_port_throughput(cores, envs_per_thread, args.steps + 0, seed=0)
        kind = "port"
        sample = ("%d envs x %d vector steps, oracle/plen_oracle.c float64, %d threads; PyBullet itself is not "
                  "installable here (SURVEY.md 8c)" % (n, args.steps, cores))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(1, args.steps), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "config5 workload (random actions U(-1,1)^18, auto-reset) on host cores; sample = %s" % sample},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def time_steps(env, acts, K, dev, flush=None):
    """K back-to-back env steps bracketed by CUDA events on the current stream -> milliseconds per step."""
    import torch
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tot = 0.0
    if flush is None:
        s0.record()
        for k in range(K):
            env.step(acts[k % len(acts)])
        s1.record()
        torch.cuda.synchronize(dev)
        return s0.elapsed_time(s1) / K
    for k in range(K):
        flush.zero_()
        s0.record()
        env.step(acts[k % len(acts)])
        s1.record()
        torch.cuda.synchronize(dev)
        tot += s0.elapsed_time(s1)
    return tot / K


def dump_index(n, dev):
    """Envs whose outputs --dump-outputs writes: all n, or DUMP_MAX_ENVS of them drawn with numpy seed 0 (ascending env
    index) when n is larger -- the same envs in every run of the same size."""
    import torch
    idx = np.arange(n) if n <= DUMP_MAX_ENVS else np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ENVS, replace=False))
    return torch.from_numpy(idx).to(dev)


def sample_step_outputs(step_out, idx):
    """float32 device copies of the rows idx of what env.step returned (obs, reward, done, info)."""
    obs, reward, done, info = step_out
    out = {"obs": obs, "reward": reward, "done": done, "timeout": info["timeout"], "terminal_obs": info["terminal_obs"]}
    return {k: v.index_select(0, idx).float() for k, v in out.items()}


def td3_leg(dev, dist, rank, world, vector_steps=24, envs=16384, batch=4096, updates_per_step=2):
    """BASELINE configs 4 / 5, the learner side: 16,384 device-resident envs per GPU feeding a device replay ring, TD3
    updates (plen_td3_*: tcgen05 3xTF32 products, minibatch 4096 per GPU) between env steps, and -- at N > 1 -- the ONE
    collective of the path family: an NCCL all-reduce (mean) of the flat gradient vectors (155,138 critic + 77,330 actor
    floats) between the gradient kernels and Adam.  Timed on the device (CUDA events), max over ranks."""
    import torch
    from plen_ml_walk_b200.sharding import env_seed, max_over_ranks
    from plen_ml_walk_b200.td3 import ReplayBuffer, TD3Agent
    from plen_ml_walk_b200.vec_env import PlenVecEnv
    torch.manual_seed(0)                                   # identical initial networks on every rank
    agent = TD3Agent(device=dev, seed=env_seed(0, rank), max_batch=batch, precision="tf32")
    env = PlenVecEnv(envs, device=dev)
    rb = ReplayBuffer(envs * (vector_steps + 8), device=dev, seed=env_seed(0, rank))
    gen = torch.Generator(device=dev); gen.manual_seed(env_seed(1, rank))
    ar_bytes = [0]

    def allreduce_mean(flat_grad):
        if dist:
            dist.all_reduce(flat_grad)
            flat_grad.mul_(1.0 / world)
            ar_bytes[0] += flat_grad.numel() * 4

    hook = allreduce_mean if dist else None                # N = 1: the whole update is one captured CUDA graph
    state = env.reset().clone()

    def one(train):
        action = torch.empty((envs, 18), device=dev).uniform_(-1, 1, generator=gen)
        obs, reward, done, info = env.step(action)
        rb.add(state, action, torch.where(done[:, None], info["terminal_obs"], obs), reward, done & ~info["timeout"])
        state.copy_(obs)
        for _ in range(updates_per_step if train else 0):
            agent.train(rb, batch, grad_hook=hook)

    for w in range(4):
        one(w >= 2)
    torch.cuda.synchronize(dev)
    if dist:
        dist.barrier()
    ar_bytes[0] = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(vector_steps):
        one(True)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = max_over_ranks(e0.elapsed_time(e1), dist, dev)
    chk = torch.stack([agent._flat[k].double().sum() for k in ("actor", "critic", "actor_target", "critic_target")])
    same = True
    if dist:
        allc = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        same = all(bool(torch.equal(c, allc[0])) for c in allc)
    n_up = vector_steps * updates_per_step
    out = {"value": world * envs * vector_steps / (ms * 1e-3), "unit": UNIT, "envs_per_gpu": envs, "vector_steps": vector_steps,
           "updates": n_up, "minibatch_per_gpu": batch, "updates_per_s": n_up / (ms * 1e-3),
           "samples_per_s": world * batch * n_up / (ms * 1e-3), "samples_per_env_step": batch * updates_per_step / envs,
           "learner_precision": "3xTF32 on tcgen05 (plen_td3_set_precision 1)",
           "allreduce": ("NCCL all-reduce (mean) of the flat gradients, %.2f MB per update, parameters identical across ranks: %s"
                         % (ar_bytes[0] / max(1, n_up) / 1e6, same)) if dist else "none (1 GPU)",
           "td3_kernel_launches": agent.kernel_launches(),
           "note": "env step + replay add + %d TD3 updates per vector step; the reference does 1 update of 100 samples per "
                   "env step (plen_td3.py:122-129), i.e. 100 samples per env-step" % updates_per_step}
    env.close(); agent.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--total-envs", type=int, default=1048576, help="config 5: envs in total, split over the GPUs (strong scaling)")
    ap.add_argument("--envs-per-gpu", type=int, default=0, help="fix the per-GPU size instead (weak scaling)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-td3-leg", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (obs, reward, done, timeout, terminal_obs; rank 0's envs) "
                         "as DIR/<name>.npy in float32, for at most %d envs (a fixed seeded sample of larger runs)" % DUMP_MAX_ENVS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    from plen_ml_walk_b200 import _abi
    from plen_ml_walk_b200.sharding import bind_host_to_gpu, env_seed, max_over_ranks
    from plen_ml_walk_b200.vec_env import PlenVecEnv

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    # N > 1: every rank runs on (and pins its host buffers next to) the CPU cores local to its GPU
    host_affinity = bind_host_to_gpu(local_rank) if world > 1 and not os.environ.get("PLEN_NO_BIND") else "unchanged"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        # NCCL_DEBUG is left as the launcher set it (the driver counts ranks from its INFO lines); the JSON line is the
        # LAST thing rank 0 prints, after the process group is gone
        import torch.distributed as dist_mod
        dist_mod.init_process_group("nccl", device_id=dev)
        dist = dist_mod

    weak = args.envs_per_gpu > 0
    E = args.envs_per_gpu if weak else args.total_envs // world
    K, W = args.steps, max(3, args.warmup)
    env = PlenVecEnv(E, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(env_seed(0, rank))
    acts = [torch.empty((E, 18), device=dev).uniform_(-1, 1, generator=gen) for _ in range(4)]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MiB > 126 MB L2
    dump_idx = dump_index(E, dev) if args.dump_outputs and rank == 0 else None
    env.reset()
    for w in range(W):
        env.step(acts[w % 4])
    torch.cuda.synchronize(dev)

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident leg (the timed region): K steps of plen_step exactly as a user calls it, each bracketed by CUDA
    #      events on the launching stream, L2 flushed in between
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.wait_first()              # nvidia-smi needs a moment before its first sample: do not let it eat the timed region
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    launches0 = env.launches
    barrier()
    t_w0 = time.time()
    for k in range(K):
        flush.zero_()
        ev[k][0].record()
        step_out = env.step(acts[k % 4])
        ev[k][1].record()
    barrier()
    t_w1 = time.time()
    launches1 = env.launches
    # copied now: the env returns reused buffers, which the steps below overwrite
    dump = sample_step_outputs(step_out, dump_idx) if dump_idx is not None else None
    # ---- per-kernel durations for the roofline: Kb MORE steps of the same workload, right behind the timed region and
    #      still under the clock sampler, with the library's CUDA-event brackets around every kernel.  They are not part of
    #      the timed region because a bracketed plen_step runs its kernels in the single-stream order (a kernel's duration
    #      is only meaningful when it has the GPU to itself), whereas the product runs two ranges of the batch concurrently.
    Kb = max(3, min(K, 10))
    env.profile_enable(Kb)
    evb = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    bracketed_ms = 0.0
    for k in range(Kb):
        flush.zero_()
        evb[0].record()
        env.step(acts[k % 4])
        evb[1].record()
        torch.cuda.synchronize(dev)
        bracketed_ms += evb[0].elapsed_time(evb[1])
    t_w2 = time.time()
    # a short run spans only a few 50 ms sampling periods: keep the SAME load on, untimed, until at least five samples
    # under load exist, and say so
    extra = 0
    while sampler.proc and sampler.count_in(t_w0, time.time()) < 5 and time.time() - t_w2 < 2.0:
        env.step(acts[extra % 4])
        torch.cuda.synchronize(dev)
        extra += 1
    clocks = sampler.stop(t_w0, time.time())
    clocks["samples_in_timed_region"] = sampler.count_in(t_w0, t_w1)
    if extra:
        clocks["note"] = "%d untimed steps of the same workload appended to collect samples under load" % extra
    gpu_launches = launches1 - launches0
    prof = env.profile_read()
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    total_ms = max_over_ranks(total_ms, dist, dev)
    value = world * E * K / (total_ms * 1e-3)
    faults = env.fault_count()

    # ---- end-to-end leg: HOST pinned buffers through plen_step_host (H2D actions, step, D2H obs/reward/done)
    Ke = max(3, min(K, 10))
    h_act = [torch.empty((E, 18), dtype=torch.float32).uniform_(-1, 1).pin_memory() for _ in range(2)]
    h_obs = torch.empty((E, 26), dtype=torch.float32).pin_memory()
    h_rew = torch.empty(E, dtype=torch.float32).pin_memory()
    h_done = torch.empty(E, dtype=torch.uint8).pin_memory()
    env.step_host(h_act[0], h_obs, h_rew, h_done)
    barrier()
    t0 = time.perf_counter()
    for k in range(Ke):
        env.step_host(h_act[k % 2], h_obs, h_rew, h_done)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_val = world * E * Ke / max_over_ranks(e2e_s, dist, dev)

    line = None
    if rank == 0:
        peak, peak_src = _peaks()
        import ctypes as C
        tf, mhz = C.c_float(), C.c_float()
        if env.lib.plen_measure_fp32_peak(local_rank, 1, C.byref(tf), C.byref(mhz)) == 0 and tf.value > 0:
            fp32_peak, fp32_src = float(tf.value), "measured live (plen_measure_fp32_peak, FFMA2 chains, best of 4); not in MEASURED_PEAKS.json"
        else:
            fp32_peak, fp32_src = FP32_NOMINAL_TFLOPS, "nominal 148 SM x 128 lanes x 2 x 1.965 GHz"
        step_ms = total_ms / K
        # dominant kernel = k_solve (one launch per physics tick over all E robots): CUDA events recorded around every
        # launch of the Kb bracketed steps by the library itself (plen_profile_enable), on the launching stream
        solve_ms = prof["ms_solve"] / max(1, prof["steps"] * TICKS_PER_STEP)
        solve_tf = E * FLOP_SOLVE_PER_ROBOT_TICK / (solve_ms * 1e-3) / 1e12
        step_tf = FLOP_PER_ENV_STEP * value / world / 1e12
        hbm_achieved = E * (BYTES_PER_ENV_STEP / TICKS_PER_STEP) / (solve_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak" if weak else "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": ("config5: %d envs in total over %d GPU(s) = %d envs/GPU, random actions U(-1,1)^18, "
                                    "auto-reset, 4 ticks/step" % (E * world, world, E)),
                       "total_envs": E * world, "envs_per_gpu": E, "l2": "256 MiB flush between timed steps",
                       "host_affinity": host_affinity},
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": E * 18 * 4,
                    "d2h_bytes_per_step": E * (26 * 4 + 4 + 1), "steps": Ke},
            "gpu_launches": gpu_launches,
            "numeric_faults": faults,
            "clocks": clocks,
            # the path is FP32-issue bound (SURVEY.md 8d), so the primary roofline is the FP32 FMA pipe; the HBM one follows
            "roofline": {"bound": "fp32", "achieved": solve_tf, "peak": fp32_peak, "unit": "TFLOP/s", "frac": solve_tf / fp32_peak,
                         "traffic": SOLVE_DRAM_BYTES_PER_ROBOT * E, "peak_source": fp32_src, "kernel": "k_solve",
                         "kernel_ms_per_launch": solve_ms, "launches_per_step": TICKS_PER_STEP,
                         "measured_over": "%d bracketed steps behind the timed region (single-stream order, kernel alone on the GPU)" % Kb,
                         "flop_per_launch": E * FLOP_SOLVE_PER_ROBOT_TICK, "flop_per_robot_tick": FLOP_SOLVE_PER_ROBOT_TICK,
                         "whole_step": {"achieved": step_tf, "frac": step_tf / fp32_peak, "flop_per_env_step": FLOP_PER_ENV_STEP,
                                        "frac_by_ncu_op_metrics_without_ffma2": FLOP_PER_ENV_STEP_NCU_OP_METRICS * value / world / 1e12 / fp32_peak},
                         "reference_algorithm": {"flop_per_env_step": REF_ALGO_FLOP_PER_ENV_STEP,
                                                 "equivalent_tflops": REF_ALGO_FLOP_PER_ENV_STEP * value / world / 1e12,
                                                 "equivalent_frac": REF_ALGO_FLOP_PER_ENV_STEP * value / world / 1e12 / fp32_peak},
                         "note": "flop = executed FADD + FMUL + 2 FFMA + 4 FFMA2 thread operations counted from the SASS execution counts of "
                                 "ncu's source page on this workload (frozen in BASELINE.md; ncu's op_ffma metric does not count the packed "
                                 "FFMA2 that is 82 % of k_solve's flops, so lines before this build quoted a 6.2x smaller solve count); "
                                 "k_solve keeps the FMA pipe 34 % busy at 2 warps per scheduler: what is left is the dependency latency of "
                                 "the Gauss-Seidel row chain; reference_algorithm = the same env-steps/s priced at the oracle's instrumented "
                                 "flop count of Bullet's ABA + velocity-space PGS; traffic = ncu DRAM bytes per robot (32768-robot capture) x robots per launch"},
            "roofline_hbm": {"bound": "hbm", "achieved": hbm_achieved, "peak": peak, "unit": "GB/s", "frac": hbm_achieved / peak,
                             "peak_source": peak_src, "kernel": "k_solve",
                             "algorithmic_bytes_per_launch": E * BYTES_PER_ENV_STEP / TICKS_PER_STEP,
                             "bytes_per_env_step": BYTES_PER_ENV_STEP, "note": "not the binding roofline of this path"},
            "kernel_ms_per_step": {"k_dyn": prof["ms_dyn"] / max(1, prof["steps"]), "k_solve": prof["ms_solve"] / max(1, prof["steps"]),
                                   "k_post": prof["ms_post"] / max(1, prof["steps"])},
            "kernel_ms_note": "CUDA-event brackets written by the library around every kernel of %d steps of the same workload run "
                              "right behind the timed region (%.3f ms per bracketed step): a bracketed plen_step runs in the "
                              "single-stream order, the timed steps run as two concurrent ranges like any user call (DESIGN.md); "
                              "k_solve includes k_rank and the rare-path k_solve_x of the tick" % (Kb, bracketed_ms / Kb),
        }
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.cpu().numpy())
        del dump
    env.close()
    del env, acts, h_act, h_obs
    torch.cuda.empty_cache()
    td3 = None
    if not args.no_td3_leg:
        td3 = td3_leg(dev, dist, rank, world)              # every rank takes part (all-reduce at N > 1)
    if rank == 0:
        if td3 is not None:
            line.setdefault("other_configs", {})["config4_td3_%s" % ("dp%d" % world if world > 1 else "1gpu")] = td3
        if world == 1 and not args.no_other_configs:
            # the other BASELINE configs that fit this run, device-resident, CUDA events, same seed discipline: round 1's
            # 131,072-env shard (weak-scaling unit; 256 MiB L2 flush between steps) and config 2 (4,096 envs, which under-fills
            # 148 SMs -- one wave of solver warps -- so it is reported next to the headline, not instead of it)
            other = {}
            for name, n2, k2, fl, note in (
                    ("config5_shard_131072_envs", 131072, 30, flush, "one of eight shards of config 5 (weak-scaling unit); L2 flushed between steps"),
                    ("config2_4096_envs", 4096, 200, None, "BASELINE configs[1]; back-to-back steps, no L2 flush (working set 28 MB)")):
                e2 = PlenVecEnv(n2, device=dev)
                a2 = [torch.empty((n2, 18), device=dev).uniform_(-1, 1, generator=gen) for _ in range(4)]
                e2.reset()
                for w in range(10):
                    e2.step(a2[w % 4])
                torch.cuda.synchronize(dev)
                ms2 = time_steps(e2, a2, k2, dev, fl)
                other[name] = {"value": n2 / (ms2 * 1e-3), "unit": UNIT, "ms_per_step": ms2, "steps": k2, "note": note}
                e2.close()
            line.setdefault("other_configs", {}).update(other)
        if not args.no_cpu_baseline and world == 1:
            cores = len(os.sched_getaffinity(0))
            probe, _, _ = cpu_port_throughput(cores, 8, 4, seed=1)
            ept = int(max(8, min(2048, probe * 0.25 / cores)))          # ~0.25 s per vector step, ~12 s in total
            v, dt, n = cpu_port_throughput(cores, ept, 48)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "%d envs x 48 vector steps (%.1f s of wall time on %d threads), "
                                              "float64 oracle port (oracle/plen_oracle.c); PyBullet itself is not "
                                              "installable here (SURVEY.md 8c)" % (n, dt, cores)}
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        sys.stdout.flush()
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
