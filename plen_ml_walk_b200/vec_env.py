"""PlenVecEnv -- the reference's Gym surface (PlenWalkEnv, plen_bullet/src/plen_bullet/plen_env.py:22-1097),
vectorised over N device-resident robots and driven through the C ABI of libplen_b200.so.

Same verbs and attributes as the reference env so plen_td3.py / walk_eval.py / trajectory_eval.py style loops port
one-to-one (SURVEY.md section 8b):

    env = PlenVecEnv(num_envs=4096, device="cuda:0")          # gym.make("PlenWalkEnv-v1")        plen_td3.py:43
    obs = env.reset()                                          # [N,26]                            plen_env.py:558
    obs, reward, done, info = env.step(actions)                # [N,26], [N], [N] bool, dict       plen_env.py:638

Differences forced by batching: `step` auto-resets finished envs in the same kernel launch (the reference leaves the
reset to the caller, plen_td3.py:122-129); `info["terminal_obs"]` holds the last observation of the finished
episodes, `info["timeout"]` the TimeLimit truncation flag (plen_td3.py:109-110 uses it as done_bool = 0).

torch is used only for device memory and streams; every computation is in the CUDA library.  No CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _abi
from .urdf_loader import PlenModel, packaged_model

OBS_DIM, ACT_DIM = 26, 18
# the observation words (plen_env.py:816-822); set_obs_noise's std / bias_std cover the first 24, contact_flip the last two
OBS_NAMES = ["q%d" % (j + 1) for j in range(18)] + ["z", "vx", "roll", "pitch", "yaw", "y", "right_contact", "left_contact"]
NOISE_WORDS = 24

# plen_env.py:148-167 (env_ranges) and :170-189 (real_ranges)
ENV_RANGES = [[-1.57, 1.57], [-0.15, 1.5], [-0.95, 0.75], [-0.9, 0.3], [-0.95, 1.2], [-0.8, 0.4],
              [-1.57, 1.57], [-1.5, 0.15], [-0.75, 0.95], [-0.3, 0.9], [-1.2, 0.95], [-0.4, 0.8],
              [-1.57, 1.57], [-0.15, 1.57], [-0.2, 0.35], [-1.57, 1.57], [-0.15, 1.57], [-0.2, 0.35]]
REAL_RANGES = [[-1.57, 1.57], [-0.15, 1.5], [-0.95, 1.2], [-1.0, 1.57], [-0.95, 1.2], [-0.8, 0.4],
               [-1.57, 1.57], [-1.5, 0.15], [-1.2, 0.95], [-1.0, 1.57], [-1.2, 1.2], [-0.4, 0.8],
               [-1.57, 1.57], [-0.15, 1.57], [-0.2, 0.35], [-1.57, 1.57], [-0.15, 1.57], [-0.2, 0.35]]


class Box:
    """Minimal stand-in for gym.spaces.Box (gym is not a dependency): low/high/shape/dtype/sample."""

    def __init__(self, low, high, dtype=np.float32, seed=None):
        self.low = np.asarray(low, dtype=dtype)
        self.high = np.asarray(high, dtype=dtype)
        self.shape = self.low.shape
        self.dtype = np.dtype(dtype)
        self._rng = np.random.default_rng(seed)

    def seed(self, seed=None):
        self._rng = np.random.default_rng(seed)

    def sample(self):
        lo = np.where(np.isfinite(self.low), self.low, -1.0)
        hi = np.where(np.isfinite(self.high), self.high, 1.0)
        return self._rng.uniform(lo, hi).astype(self.dtype)


def _spaces():
    # plen_env.py:141-144 (action space) and :246-263 (observation space)
    lo = [r[0] for r in ENV_RANGES] + [0, -np.inf, -np.pi, -np.pi, -np.pi, -np.inf, 0, 0]
    hi = [r[1] for r in ENV_RANGES] + [0.25, np.inf, np.pi, np.pi, np.pi, np.inf, 1, 1]
    return Box(-np.ones(ACT_DIM), np.ones(ACT_DIM)), Box(lo, hi)


class PlenVecEnv:
    metadata = {"render.modes": []}

    def __init__(self, num_envs, device="cuda:0", joint_act=False, auto_reset=True, model: PlenModel | None = None,
                 config_overrides: dict | None = None, seed=None):
        if not torch.cuda.is_available():
            raise RuntimeError("PlenVecEnv needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _abi.load_library()
        self.device = torch.device(device)
        self.device_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.num_envs = int(num_envs)
        self.joint_act = bool(joint_act)
        self.model = model if model is not None else packaged_model()
        self._cmodel = _abi.model_to_c(self.model)
        self.cfg = _abi.PlenConfigC()
        self.lib.plen_default_config(C.byref(self.cfg), int(joint_act))
        self.cfg.auto_reset = int(auto_reset)
        if model is not None:
            self.cfg.hull_margin = float(getattr(model, "foot_margin", self.cfg.hull_margin))      # box feet carry no margin
        for k, v in (config_overrides or {}).items():
            setattr(self.cfg, k, v)
        self._ctx = self.lib.plen_create(C.byref(self.cfg), C.byref(self._cmodel), self.num_envs, self.device_index)
        if not self._ctx:
            raise RuntimeError("plen_create failed: %s" % self.lib.plen_last_error(None).decode())
        self.action_space, self.observation_space = _spaces()
        self.action_space.seed(seed)
        self.env_ranges, self.real_ranges = ENV_RANGES, REAL_RANGES
        self._max_episode_steps = int(self.cfg.max_episode_steps)         # TimeLimit attribute, plen_td3.py:110
        n, dev = self.num_envs, self.device
        self._obs = torch.empty((n, OBS_DIM), dtype=torch.float32, device=dev)
        self._terminal_obs = torch.zeros((n, OBS_DIM), dtype=torch.float32, device=dev)
        self._reward = torch.empty(n, dtype=torch.float32, device=dev)
        self._done = torch.empty(n, dtype=torch.uint8, device=dev)
        self._timeout = torch.empty(n, dtype=torch.uint8, device=dev)
        self._scales = {}                                                  # per-env scales set so far (set_env_scales)
        self._noise_on = False                                             # set_obs_noise called (and not cleared)
        self._clean_obs = self._clean_terminal_obs = None

    # ---- plumbing
    def _check(self, rc):
        if rc != 0:
            raise RuntimeError("libplen_b200: %s" % self.lib.plen_last_error(self._ctx).decode())

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @staticmethod
    def _p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def _dev_f32(self, x, shape):
        t = torch.as_tensor(x, dtype=torch.float32, device=self.device).contiguous()
        if tuple(t.shape) != tuple(shape):
            raise ValueError("expected shape %s, got %s" % (shape, tuple(t.shape)))
        return t

    # ---- Gym surface
    def seed(self, seed=None):
        """The reference env is effectively unseeded (it only defines _seed, plen_env.py:28-32); seeds action_space."""
        self.action_space.seed(seed)
        return [seed]

    def reset(self, mask=None):
        """PlenWalkEnv.reset (plen_env.py:558-614) for all envs, or for those where mask is True."""
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_reset(self._ctx, self._p(m), self._p(self._obs), self._stream()))
        return self._obs

    @property
    def launches(self):
        """Kernels of ours launched by step()/step_host()/reset()/tick() so far, counted where they are launched (bench.py reports it)."""
        return int(self.lib.plen_kernel_launches(self._ctx))

    def step(self, actions):
        """PlenWalkEnv.step (plen_env.py:638-692) for all N envs in one launch.  Returned tensors are reused buffers."""
        a = self._dev_f32(actions, (self.num_envs, ACT_DIM))
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_step(self._ctx, self._p(a), self._p(self._obs), self._p(self._reward),
                                           self._p(self._done), self._p(self._timeout), self._p(self._terminal_obs),
                                           self._stream()))
        info = {"terminal_obs": self._terminal_obs, "timeout": self._timeout.bool()}
        if self._noise_on:
            info["clean_obs"], info["clean_terminal_obs"] = self.clean_obs()
        return self._obs, self._reward, self._done.bool(), info

    def step_host(self, actions_host, obs_host, reward_host, done_host, timeout_host=None):
        """End-to-end call with HOST (ideally pinned) numpy/torch CPU buffers: H2D + step + D2H + sync."""
        def hp(x):
            if x is None:
                return None
            return C.c_void_p(x.data_ptr() if isinstance(x, torch.Tensor) else x.ctypes.data)
        self._check(self.lib.plen_step_host(self._ctx, hp(actions_host), hp(obs_host), hp(reward_host), hp(done_host),
                                            hp(timeout_host)))

    def fault_count(self):
        """Robots retired by the numeric guard (non-finite physical state -> done, reward -100, forced reset) so far."""
        c = C.c_ulonglong()
        self._check(self.lib.plen_fault_count(self._ctx, C.byref(c)))
        return int(c.value)

    def profile_enable(self, max_steps):
        """Record CUDA events around every kernel of the next max_steps step() calls (bench.py's roofline leg)."""
        self._check(self.lib.plen_profile_enable(self._ctx, int(max_steps)))

    def profile_read(self):
        """-> dict(ms_dyn, ms_solve, ms_post, steps): summed device time per kernel family since the last read."""
        d, s, p, n = C.c_float(), C.c_float(), C.c_float(), C.c_int()
        self._check(self.lib.plen_profile_read(self._ctx, C.byref(d), C.byref(s), C.byref(p), C.byref(n)))
        return {"ms_dyn": d.value, "ms_solve": s.value, "ms_post": p.value, "steps": n.value}

    def close(self):
        if getattr(self, "_ctx", None):
            self.lib.plen_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- state access (parity tests, checkpointing)
    def get_state(self):
        n, dev = self.num_envs, self.device
        qpos = torch.empty((n, 25), dtype=torch.float32, device=dev)
        qvel = torch.empty((n, 24), dtype=torch.float32, device=dev)
        aux = torch.empty((n, _abi.AUX_WORDS), dtype=torch.float32, device=dev)
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_get_state(self._ctx, self._p(qpos), self._p(qvel), self._p(aux), self._stream()))
        return qpos, qvel, aux

    def set_state(self, qpos=None, qvel=None, aux=None):
        n = self.num_envs
        qpos = None if qpos is None else self._dev_f32(qpos, (n, 25))
        qvel = None if qvel is None else self._dev_f32(qvel, (n, 24))
        aux = None if aux is None else self._dev_f32(aux, (n, _abi.AUX_WORDS))
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_set_state(self._ctx, self._p(qpos), self._p(qvel), self._p(aux), self._stream()))

    def get_manifold(self):
        """Persistent sole manifolds [N, 52] (config_overrides={"sole_manifold": 1} only; layout: include/plen_b200.h)."""
        man = torch.empty((self.num_envs, _abi.MAN_WORDS), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_get_manifold(self._ctx, self._p(man), self._stream()))
        return man

    def set_manifold(self, man):
        man = self._dev_f32(man, (self.num_envs, _abi.MAN_WORDS))
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_set_manifold(self._ctx, self._p(man), self._stream()))

    def set_env_scales(self, friction=None, motor_force=None, motor_gain=None):
        """Per-env domain randomisation (SURVEY.md 8f-3): scale factors [N] of the foot friction coefficients, the servo force
        limit and the servo position gain; None leaves a quantity unchanged, 1.0 is the reference's constant.

        Resets: by default a reset (explicit or in-kernel auto-reset) restores the ONE post-reset snapshot that was settled for
        8 ticks under unit scales at creation, whatever the robot's own scales are; its first steps then run under its scales.
        Call settle_resets() after the setters to settle every robot's reset state under its own scales instead."""
        arr = [None if x is None else self._dev_f32(x, (self.num_envs,)) for x in (friction, motor_force, motor_gain)]
        for k, x in zip(("friction", "motor_force", "motor_gain"), arr):
            if x is not None:
                self._scales[k] = x.clone()               # mirror kept for save_state (the library has no getter)
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_set_env_scales(self._ctx, *[self._p(x) for x in arr], self._stream()))

    @property
    def body_links(self):
        """Names of the URDF links folded into each of the 19 bodies of set_env_mass: body 0 is the torso composite, body 1 + j
        the body moved by joint j (action order)."""
        return [list(self.model.body_links[0])] + [list(self.model.body_links[l]) for l in range(6, 24)]

    def set_env_mass(self, mass_scale=None, payload=None):
        """Per-env mass randomisation (SURVEY.md 8f-3).  None leaves a part unchanged.

        mass_scale: [N] (one factor for every body) or [N,19]: factor on the mass and the rotational inertia of each body
                    (uniform density scaling, centre of mass unchanged); the bodies are listed in body_links.
        payload:    [N,4] (m, x, y, z): a point mass of m kg rigidly attached at (x, y, z) in the torso body frame (the frame of
                    the base pose in get_state's qpos), without rotational inertia of its own.
        Raises ValueError on a wrong shape, a scale that is not finite and > 0, or a payload that is not finite or has m < 0.
        Before the first call every robot has scale 1 and payload 0, and such a robot steps bit-identically to a context that
        never called this.  Takes effect from the next tick.

        Resets, as for set_env_scales: by default a reset (explicit or in-kernel auto-reset) restores the ONE post-reset
        snapshot settled under the nominal model at creation, and the robot's own masses apply from its first tick after that.
        Call settle_resets() after the setters to settle every robot's reset state under its own masses instead."""
        n = self.num_envs
        s = p = None
        if mass_scale is not None:
            s = torch.as_tensor(mass_scale, dtype=torch.float32, device=self.device)
            if tuple(s.shape) == (n,):
                s = s[:, None].expand(n, _abi.BODIES)
            s = self._dev_f32(s, (n, _abi.BODIES))
            if not bool(torch.isfinite(s).all()) or not bool((s > 0).all()):
                raise ValueError("mass_scale must be finite and > 0")
        if payload is not None:
            p = self._dev_f32(payload, (n, 4))
            if not bool(torch.isfinite(p).all()) or not bool((p[:, 0] >= 0).all()):
                raise ValueError("payload must be finite with a mass >= 0")
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_set_env_mass(self._ctx, self._p(s), self._p(p), self._stream()))

    def _get_env_mass(self):
        n, dev = self.num_envs, self.device
        s = torch.empty((n, _abi.BODIES), dtype=torch.float32, device=dev)
        p = torch.empty((n, 4), dtype=torch.float32, device=dev)
        with torch.cuda.device(self.device):
            rc = self.lib.plen_get_env_mass(self._ctx, self._p(s), self._p(p), self._stream())
        if rc < 0:
            self._check(rc)
        return s, p, rc == 1

    def get_env_mass(self):
        """-> (mass_scale [N,19], payload [N,4]) as the device holds them (1 and 0 where set_env_mass was never called)."""
        s, p, _ = self._get_env_mass()
        return s, p

    @property
    def max_latency_ticks(self):
        """Largest command delay set_env_latency accepts: 2 * substeps physics ticks (8 ticks, 33 ms at the defaults)."""
        return _abi.MAX_LATENCY_STEPS * int(self.cfg.substeps)

    def set_env_latency(self, ticks, history=None):
        """Per-env servo command latency (SURVEY.md 8f-3): each robot's servos act on its commands `ticks` physics ticks late.

        ticks:   an int (every robot) or [N] integers, 0 <= d <= max_latency_ticks; one tick is 1/240 s = 4.17 ms at the default
                 rate.  Tick k of a step (0 <= k < substeps) applies the raw servo targets of the step ceil(max(d - k, 0) /
                 substeps) steps back: 0 is the stock behaviour, d = substeps applies the previous step's command for the
                 whole step.  A command from before the robot's last reset (explicit or auto-reset) is the reset-pose hold
                 target 0 rad.
        history: [N,2,18] raw targets of the last step and of the step before (radians, relative to the robots' current
                 episode counters), None to keep the recorded ones; load_state uses it to continue a run bit for bit.
        Raises ValueError on a wrong shape, a non-integer, a negative value or a value above max_latency_ticks.
        The first call starts a command history seeded with each robot's last servo targets, as if they had been held;
        every step() / step_host() records into it from then on.  Delays may change between any two steps.  tick() and
        debug_dynamics() are raw physics and ignore the latency."""
        n = self.num_envs
        t = torch.as_tensor(ticks, device=self.device)
        if t.dim() == 0:
            t = t.expand(n)
        if tuple(t.shape) != (n,):
            raise ValueError("ticks: expected an int or shape (%d,), got %s" % (n, tuple(t.shape)))
        if t.dtype.is_floating_point:
            if not bool(torch.isfinite(t).all()) or not bool((t == torch.round(t)).all()):
                raise ValueError("ticks must be integers")
        elif t.dtype == torch.bool or t.dtype.is_complex:
            raise ValueError("ticks must be integers")
        if not bool((t >= 0).all()) or not bool((t <= self.max_latency_ticks).all()):
            raise ValueError("ticks must lie in 0 .. %d (2 * substeps)" % self.max_latency_ticks)
        t = t.to(torch.int32).contiguous()
        h = None if history is None else self._dev_f32(history, (n, 2, ACT_DIM))
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_set_env_latency(self._ctx, self._p(t), self._p(h), self._stream()))

    def _get_env_latency(self):
        n, dev = self.num_envs, self.device
        t = torch.empty(n, dtype=torch.int32, device=dev)
        h = torch.empty((n, 2, ACT_DIM), dtype=torch.float32, device=dev)
        with torch.cuda.device(self.device):
            rc = self.lib.plen_get_env_latency(self._ctx, self._p(t), self._p(h), self._stream())
        if rc < 0:
            self._check(rc)
        return t, h, rc == 1

    def get_env_latency(self):
        """-> int32 [N]: each robot's command delay in physics ticks (0 where set_env_latency was never called)."""
        return self._get_env_latency()[0]

    def settle_resets(self, start_pose=None):
        """Per-env reset states (no reference counterpart): run the reference's reset procedure (plen_env.py:558-574) for every
        robot under its current friction / force / gain scales and masses, and make the result the state that robot's resets
        (reset(), the in-kernel auto-reset, the numeric guard) restore from now on.

        start_pose: None (the reference's start position, heading 0), [4] for every robot or [N,4]: (x, y, z, yaw) -- base
                    position in the world (m) and heading about world z (rad).  Each robot is teleported there with zero
                    joints, velocities and targets, empty contact caches, and settled for reset_ticks (8) ticks with hold
                    target 0.  Raises ValueError on a wrong shape or a non-finite value.
        Intended workflow: set the domain-randomisation parameters (set_env_scales, set_env_mass), call settle_resets(), then
        reset() if the robots should start from their new reset states now -- the running states are not touched, a new
        reset state applies from each robot's next reset.  Command latency does not act during the settle (raw physics, like
        tick()).  A nominal robot settled from the default pose gets exactly the shared snapshot."""
        n = self.num_envs
        p = None
        if start_pose is not None:
            p = torch.as_tensor(start_pose, dtype=torch.float32, device=self.device)
            if tuple(p.shape) == (4,):
                p = p[None, :].expand(n, 4)
            p = self._dev_f32(p, (n, 4))
            if not bool(torch.isfinite(p).all()):
                raise ValueError("start_pose must be finite")
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_settle_env_resets(self._ctx, self._p(p), self._stream()))

    def set_env_resets(self, qpos=None, qvel=None, aux=None, man=None):
        """User-supplied reset states (recorded states, curricula) in the layouts of set_state / set_manifold; None leaves that
        part of every robot's reset state as it is (the shared snapshot before the first settle_resets / set_env_resets).  The
        observation of each reset state is computed from it.  man needs config_overrides={"sole_manifold": 1}."""
        n = self.num_envs
        qpos = None if qpos is None else self._dev_f32(qpos, (n, 25))
        qvel = None if qvel is None else self._dev_f32(qvel, (n, 24))
        aux = None if aux is None else self._dev_f32(aux, (n, _abi.AUX_WORDS))
        man = None if man is None else self._dev_f32(man, (n, _abi.MAN_WORDS))
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_set_env_resets(self._ctx, self._p(qpos), self._p(qvel), self._p(aux), self._p(man),
                                                     self._stream()))

    def _get_env_resets(self):
        n, dev = self.num_envs, self.device
        qpos = torch.empty((n, 25), dtype=torch.float32, device=dev)
        qvel = torch.empty((n, 24), dtype=torch.float32, device=dev)
        aux = torch.empty((n, _abi.AUX_WORDS), dtype=torch.float32, device=dev)
        obs = torch.empty((n, OBS_DIM), dtype=torch.float32, device=dev)
        man = torch.empty((n, _abi.MAN_WORDS), dtype=torch.float32, device=dev) if int(self.cfg.sole_manifold) else None
        with torch.cuda.device(self.device):
            rc = self.lib.plen_get_env_resets(self._ctx, self._p(qpos), self._p(qvel), self._p(aux), self._p(obs), self._p(man),
                                              self._stream())
        if rc < 0:
            self._check(rc)
        return (qpos, qvel, aux, obs, man), rc == 1

    def get_env_resets(self):
        """-> (qpos [N,25], qvel [N,24], aux [N,29], obs [N,26], man [N,52] or None without sole_manifold): the state each
        robot's next reset restores (the shared snapshot where no settle_resets / set_env_resets has been called)."""
        return self._get_env_resets()[0]

    def clear_env_resets(self):
        """Drop the per-env reset states: every reset restores the shared snapshot again, exactly as on a fresh env."""
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_clear_env_resets(self._ctx, self._stream()))

    def _noise_param(self, x, name):
        """float, [24], [N] or [N,24] (a 1-D [24] is per word, also when N == 24) -> [N,24] float32 on the device"""
        n = self.num_envs
        t = torch.as_tensor(x, dtype=torch.float32, device=self.device)
        if t.dim() == 0:
            t = t.expand(n, NOISE_WORDS)
        elif tuple(t.shape) == (NOISE_WORDS,):
            t = t[None, :].expand(n, NOISE_WORDS)
        elif tuple(t.shape) == (n,):
            t = t[:, None].expand(n, NOISE_WORDS)
        if tuple(t.shape) != (n, NOISE_WORDS):
            raise ValueError("%s: expected a float, (%d,), (%d,) or (%d, %d), got %s" % (name, NOISE_WORDS, n, n, NOISE_WORDS,
                                                                                       tuple(t.shape)))
        if not bool(torch.isfinite(t).all()) or not bool((t >= 0).all()):
            raise ValueError("%s must be finite and >= 0" % name)
        return t.contiguous()

    def set_obs_noise(self, std=None, bias_std=None, contact_flip=None, seed=None, first_env_id=None):
        """Per-env observation noise (SURVEY.md 8f-3, sensing side): what step() / step_host() / reset() return as obs and
        info["terminal_obs"] carries sensor noise; reward, done, the gait counters and the physics keep the true state.

        std:          white noise sigma of the 24 continuous words (OBS_NAMES[:24]: q1..q18 rad, z m, vx m/s, roll / pitch /
                      yaw rad, y m): a float, [24] (per word), [N] (per robot) or [N,24].  Fresh N(0, sigma^2) every observation.
        bias_std:     the same shapes: std of a per-episode bias b = bias_std * N(0,1), drawn at every reset of the robot and
                      constant over its episode (IMU offset, servo zero error).  Episodes running at the first call keep b = 0.
        contact_flip: a float or [N]: probability that each contact flag (OBS_NAMES[24:]) reads 1 - flag.
        seed:         of the counter-based draws (default: the current one, 0 at the first call).
        first_env_id: global id of robot 0 (default: the current one, 0): a shard of a larger population passes its first
                      robot's id and draws the noise that robot would get in one big env.
        None leaves a part unchanged (zero at the first call).  Words with std = bias = 0 are passed through bit for bit.  No
        clipping or angle wrapping is applied.  Raises ValueError on a wrong shape, a non-finite or negative std, a
        contact_flip outside [0, 1], or a negative first_env_id.  While noise is on, step() adds info["clean_obs"] and
        info["clean_terminal_obs"] (clean_obs()).  The draws advance with a counter on the device, so a captured CUDA graph
        of step() draws new noise on every replay."""
        n = self.num_envs
        s = None if std is None else self._noise_param(std, "std")
        b = None if bias_std is None else self._noise_param(bias_std, "bias_std")
        f = None
        if contact_flip is not None:
            f = torch.as_tensor(contact_flip, dtype=torch.float32, device=self.device)
            if f.dim() == 0:
                f = f.expand(n)
            f = self._dev_f32(f, (n,))
            if not bool(torch.isfinite(f).all()) or not bool(((f >= 0) & (f <= 1)).all()):
                raise ValueError("contact_flip must lie in [0, 1]")
        _, cur_seed, cur_first = self._get_obs_noise_params()
        seed = cur_seed if seed is None else int(seed)
        first = cur_first if first_env_id is None else int(first_env_id)
        if not 0 <= seed < 2 ** 64:
            raise ValueError("seed must lie in 0 .. 2^64 - 1")
        if first < 0:
            raise ValueError("first_env_id must be >= 0")
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_set_env_obs_noise(self._ctx, self._p(s), self._p(b), self._p(f), C.c_ulonglong(seed),
                                                        C.c_longlong(first), self._stream()))
        self._noise_on = True
        if self._clean_obs is None:     # allocated here, not inside a step that may be under CUDA graph capture
            self._clean_obs = torch.zeros((n, OBS_DIM), dtype=torch.float32, device=self.device)
            self._clean_terminal_obs = torch.zeros((n, OBS_DIM), dtype=torch.float32, device=self.device)

    def _get_obs_noise_params(self):
        seed, first = C.c_ulonglong(), C.c_longlong()
        rc = self.lib.plen_get_env_obs_noise(self._ctx, None, None, None, None, None, C.byref(seed), C.byref(first), self._stream())
        if rc < 0:
            self._check(rc)
        return rc == 1, int(seed.value), int(first.value)

    def get_obs_noise(self):
        """-> dict(std [N,24], bias_std [N,24], contact_flip [N], bias [N,24] of the running episodes, counter [N] int32
        (the draw counters' uint32 bits), seed, first_env_id, active); zeros where set_obs_noise was never called."""
        n, dev = self.num_envs, self.device
        s, b, bias = (torch.empty((n, NOISE_WORDS), dtype=torch.float32, device=dev) for _ in range(3))
        f = torch.empty(n, dtype=torch.float32, device=dev)
        c = torch.empty(n, dtype=torch.int32, device=dev)
        seed, first = C.c_ulonglong(), C.c_longlong()
        with torch.cuda.device(self.device):
            rc = self.lib.plen_get_env_obs_noise(self._ctx, self._p(s), self._p(b), self._p(f), self._p(bias), self._p(c),
                                                 C.byref(seed), C.byref(first), self._stream())
        if rc < 0:
            self._check(rc)
        return {"std": s, "bias_std": b, "contact_flip": f, "bias": bias, "counter": c, "seed": int(seed.value),
                "first_env_id": int(first.value), "active": rc == 1}

    def set_obs_noise_state(self, bias=None, counter=None):
        """The running per-episode biases [N,24] and draw counters [N] (uint32 bits, as get_obs_noise returns them); for
        snapshots that continue a noisy run bit for bit.  Needs set_obs_noise first."""
        n = self.num_envs
        b = None if bias is None else self._dev_f32(bias, (n, NOISE_WORDS))
        c = None
        if counter is not None:
            c = torch.as_tensor(counter, device=self.device)
            if tuple(c.shape) != (n,):
                raise ValueError("counter: expected shape (%d,), got %s" % (n, tuple(c.shape)))
            c = c.to(torch.int32).contiguous() if c.dtype != torch.int64 else \
                torch.where(c >= 2 ** 31, c - 2 ** 32, c).to(torch.int32).contiguous()
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_set_env_obs_noise_state(self._ctx, self._p(b), self._p(c), self._stream()))

    def clear_obs_noise(self):
        """Switch the observation noise off: the env is exactly the stock path again."""
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_clear_env_obs_noise(self._ctx, self._stream()))
        self._noise_on = False

    def clean_obs(self):
        """-> (obs [N,26], terminal_obs [N,26]): the noise-free observations of the last step or reset, and the noise-free
        terminal observations (written where a step reported done).  Reused buffers.  Needs set_obs_noise."""
        if self._clean_obs is None:
            raise RuntimeError("clean_obs: observation noise is off (call set_obs_noise first); obs is the clean observation")
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_get_clean_obs(self._ctx, self._p(self._clean_obs), self._p(self._clean_terminal_obs),
                                                    self._stream()))
        return self._clean_obs, self._clean_terminal_obs

    def save_state(self, path):
        """Snapshot of every env (pose, velocities, contact cache, env bookkeeping, per-env scales, masses, command delays,
        command history, reset states and observation noise) to one .pt file (SURVEY.md 8f-4)."""
        qpos, qvel, aux = self.get_state()
        ms, mp, mass_set = self._get_env_mass()
        lt, lh, lat_set = self._get_env_latency()
        rows, rows_set = self._get_env_resets()
        nz = self.get_obs_noise()
        torch.save({"num_envs": self.num_envs, "joint_act": self.joint_act, "qpos": qpos.cpu(), "qvel": qvel.cpu(), "aux": aux.cpu(),
                    "scales": {k: v.cpu() for k, v in self._scales.items()},
                    "mass": {"scale": ms.cpu(), "payload": mp.cpu()} if mass_set else None,
                    "latency": {"ticks": lt.cpu(), "history": lh.cpu()} if lat_set else None,
                    "resets": dict(zip(("qpos", "qvel", "aux", "man"), (None if t is None else t.cpu() for t in rows[:3] + rows[4:])))
                    if rows_set else None,
                    "obs_noise": {k: (v.cpu() if isinstance(v, torch.Tensor) else v) for k, v in nz.items()} if nz["active"] else None,
                    "manifold": self.get_manifold().cpu() if int(self.cfg.sole_manifold) else None}, path)

    def load_state(self, path):
        """Restore a save_state snapshot; stepping on from it reproduces the original run bit for bit."""
        d = torch.load(path, map_location="cpu")
        if int(d["num_envs"]) != self.num_envs or bool(d["joint_act"]) != self.joint_act:
            raise ValueError("snapshot is for %d envs (joint_act=%s)" % (d["num_envs"], d["joint_act"]))
        self.set_state(d["qpos"], d["qvel"], d["aux"])
        if d.get("manifold") is not None:
            self.set_manifold(d["manifold"])
        sc = d.get("scales", {})
        if sc or self._scales:      # per-env scales travel with the snapshot; a snapshot without any restores the unit scales
            ones = torch.ones(self.num_envs)
            self.set_env_scales(*[sc.get(k, ones) for k in ("friction", "motor_force", "motor_gain")])
        mass = d.get("mass")
        if mass is not None:        # per-env masses likewise; a snapshot without them restores unit values if the context had some
            self.set_env_mass(mass["scale"], mass["payload"])
        elif self._get_env_mass()[2]:
            self.set_env_mass(torch.ones(self.num_envs, _abi.BODIES), torch.zeros(self.num_envs, 4))
        lat = d.get("latency")
        if lat is not None:         # after set_state: the history is written relative to the restored episode counters
            self.set_env_latency(lat["ticks"], lat["history"])
        elif self._get_env_latency()[2]:
            self.set_env_latency(0)
        rows = d.get("resets")
        if rows is not None:        # reset states likewise; a snapshot without them leaves the context on the shared snapshot
            self.set_env_resets(rows["qpos"], rows["qvel"], rows["aux"], rows["man"])
        else:
            self.clear_env_resets()
        nz = d.get("obs_noise")
        if nz is not None:          # parameters, running biases and draw counters: the noisy run continues bit for bit
            self.set_obs_noise(nz["std"], nz["bias_std"], nz["contact_flip"], seed=nz["seed"], first_env_id=nz["first_env_id"])
            self.set_obs_noise_state(nz["bias"], nz["counter"])
        else:
            self.clear_obs_noise()

    def tick(self, targets, n_ticks=1):
        """Raw physics: n_ticks of 1/240 s with joint targets in radians, no env logic (move_joints + stepSimulation)."""
        t = self._dev_f32(targets, (self.num_envs, ACT_DIM))
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_tick(self._ctx, self._p(t), int(n_ticks), self._stream()))

    def debug_records(self):
        """Raw per-env state records [N,96] (word 79 = PGS iterations of the last tick)."""
        rec = torch.empty((self.num_envs, _abi.STATE_WORDS), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_debug_records(self._ctx, self._p(rec), self._stream()))
        return rec

    def debug_dynamics(self):
        n, dev = self.num_envs, self.device
        minv = torch.zeros((n, 24, 24), dtype=torch.float32, device=dev)
        pos = torch.zeros((n, 24, 3), dtype=torch.float32, device=dev)
        rot = torch.zeros((n, 24, 3, 3), dtype=torch.float32, device=dev)
        with torch.cuda.device(self.device):
            self._check(self.lib.plen_debug_dynamics(self._ctx, self._p(minv), self._p(pos), self._p(rot), self._stream()))
        return minv, pos, rot


class PlenWalkEnv:
    """1-env adapter with the reference's exact call shapes: reset() -> np[26]; step(a[18]) -> (obs, r, done, {}).

    Mirrors `gym.make("PlenWalkEnv-v1", render=False, joint_act=...)` (plen_env.py:15-19, :34) including the
    TimeLimit(500) wrapper; like the reference it does NOT auto-reset (the caller does, plen_td3.py:122-129).
    """

    def __init__(self, render=False, realtime=False, joint_act=False, device="cuda:0", config_overrides=None):
        if render or realtime:
            raise NotImplementedError("the B200 env is headless (PyBullet GUI / realtime modes are out of scope)")
        # config_overrides: plen_config fields, e.g. {"sole_manifold": 1} (gym.make passes keyword arguments through)
        self.vec = PlenVecEnv(1, device=device, joint_act=joint_act, auto_reset=False, config_overrides=config_overrides)
        self.action_space, self.observation_space = self.vec.action_space, self.vec.observation_space
        self.env_ranges, self.real_ranges = ENV_RANGES, REAL_RANGES
        self._max_episode_steps = self.vec._max_episode_steps
        self.joint_act = joint_act

    def seed(self, seed=None):
        return self.vec.seed(seed)

    def reset(self):
        return self.vec.reset()[0].cpu().numpy().astype(np.float64)

    def step(self, action):
        a = np.asarray(action, dtype=np.float32).reshape(1, ACT_DIM)
        obs, r, d, info = self.vec.step(a)
        return obs[0].cpu().numpy().astype(np.float64), float(r[0]), bool(d[0]), {"timeout": bool(info["timeout"][0])}

    def close(self):
        self.vec.close()
