"""Shared numpy reference of the per-robot command latency schedule (plen_set_env_latency, PlenVecEnv.set_env_latency):
which step's raw servo targets each physics tick applies.  Used by the CPU tests (warp emulation) and the GPU tests."""
import numpy as np


def latency_source(d, k, S, ep_t):
    """Source step of tick k (0 <= k < S) of an env step under a delay of d ticks: s = ceil(max(d - k, 0) / S) steps back, or -1
    when that step lies before the robot's last reset (s > ep_t, the robot's episode counter at this step), whose command is
    the reset-pose hold target 0.  Works elementwise on arrays."""
    d, ep_t = np.asarray(d, dtype=np.int64), np.asarray(ep_t, dtype=np.int64)
    late = np.maximum(d - k, 0)
    s = (late + S - 1) // S
    return np.where((s == 0) | (s <= ep_t), s, -1)


class CommandSchedule:
    """Per-tick servo targets of n robots under command latency, step by step.

    `last` [n,18] seeds the history (the raw targets of the last step and of the step before), as the first setter call does
    with the robots' last servo targets.  step(raw, d, ep_t) takes the raw targets [n,18] of the new step, the delays [n] and
    the episode counters [n] at this step, and returns the targets [S,n,18] each tick applies."""

    def __init__(self, n, S, last=None):
        self.S = S
        last = np.zeros((n, 18), dtype=np.float32) if last is None else np.asarray(last, dtype=np.float32)
        self.prev = [last.copy(), last.copy()]       # [0]: the last step, [1]: the step before

    def step(self, raw, d, ep_t):
        raw = np.asarray(raw, dtype=np.float32)
        out = np.empty((self.S,) + raw.shape, dtype=np.float32)
        for k in range(self.S):
            s = latency_source(d, k, self.S, ep_t)[:, None]
            out[k] = np.where(s == 0, raw, np.where(s == 1, self.prev[0], np.where(s == 2, self.prev[1], np.float32(0))))
        self.prev = [raw.copy(), self.prev[0]]
        return out
