"""Device-resident TD3 for the batched PLEN env -- host mirror of plen_ros/src/plen_ros_helpers/td3.py (Actor :19-57,
Critic :60-117, ReplayBuffer :122-193, TD3Agent :196-376) as driven by plen_bullet/src/plen_td3.py.

Same class / method / state_dict names as the reference so its checkpoints (`plen_bullet/models/*_actor`, `*_critic`:
keys fc1..fc3 / fc1..fc6) load unchanged.  What runs where:

  * ReplayBuffer      hand-written CUDA ring in libplen_b200.so (plen_replay_*): [capacity, 72] floats in HBM,
                      vectorised add of N transitions per call, uniform sampling with replacement on the device
                      (the reference rebuilds O(B^2) host tensors per sample, td3.py:178-191).
  * select_action     hand-written CUDA fused 3-layer MLP (plen_actor_forward), fp32, N observations per launch,
                      optional exploration noise + clip (plen_td3.py:101-104) in the same kernel.
  * train             the reference's update rule (td3.py:259-356) as hand-written CUDA (csrc/plen_td3_learn.cu): strided
                      fp32 GEMM kernel with fused bias / ReLU / tanh / mask / bias-gradient epilogues, fused Adam, fused
                      Polyak update over flat parameter vectors; 18 kernels per critic step, 36 with the policy step,
                      replayed as one CUDA graph per update, no host sync.  train_torch = the same rule in PyTorch (test reference only).

No CPU fallback for the CUDA pieces.
"""
from __future__ import annotations

import copy
import ctypes as C

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _abi

STATE_DIM, ACTION_DIM = 26, 18


class Actor(nn.Module):                                    # td3.py:19-57
    def __init__(self, state_dim=STATE_DIM, action_dim=ACTION_DIM, max_action=1.0):
        super().__init__()
        self.fc1 = nn.Linear(state_dim, 256)
        self.fc2 = nn.Linear(256, 256)
        self.fc3 = nn.Linear(256, action_dim)
        self.max_action = max_action

    def forward(self, state):
        a = F.relu(self.fc1(state))
        a = F.relu(self.fc2(a))
        return self.max_action * torch.tanh(self.fc3(a))


class Critic(nn.Module):                                   # td3.py:60-117
    def __init__(self, state_dim=STATE_DIM, action_dim=ACTION_DIM):
        super().__init__()
        self.fc1 = nn.Linear(state_dim + action_dim, 256)
        self.fc2 = nn.Linear(256, 256)
        self.fc3 = nn.Linear(256, 1)
        self.fc4 = nn.Linear(state_dim + action_dim, 256)
        self.fc5 = nn.Linear(256, 256)
        self.fc6 = nn.Linear(256, 1)

    def forward(self, state, action):
        sa = torch.cat([state, action], 1)
        q1 = self.fc3(F.relu(self.fc2(F.relu(self.fc1(sa)))))
        q2 = self.fc6(F.relu(self.fc5(F.relu(self.fc4(sa)))))
        return q1, q2

    def Q1(self, state, action):
        sa = torch.cat([state, action], 1)
        return self.fc3(F.relu(self.fc2(F.relu(self.fc1(sa)))))


_tc_checked = False


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def actor_forward(actor: Actor, obs: torch.Tensor, noise_std: float = 0.0, seed: int = 0, out: torch.Tensor | None = None,
                  precision: str = "fp32"):
    """Actor.forward for obs [N,26] (float32, CUDA) through the fused CUDA kernel; optional exploration noise + clip.
    precision "fp32": CUDA-core kernel, 1e-5 parity with the reference; "fp16": tcgen05 tensor-core kernel (FP16 operands,
    FP32 accumulation in TMEM), mean action error ~5e-4 against fp32 -- the throughput path for rollouts."""
    if not obs.is_cuda:
        raise RuntimeError("plen_actor_forward needs CUDA tensors; there is no CPU fallback")
    lib = _abi.load_library()
    obs = obs.contiguous().float()
    n = obs.shape[0]
    if out is None:
        out = torch.empty((n, ACTION_DIM), dtype=torch.float32, device=obs.device)
    w = [actor.fc1.weight, actor.fc1.bias, actor.fc2.weight, actor.fc2.bias, actor.fc3.weight, actor.fc3.bias]
    w = [t.detach().contiguous() for t in w]
    if tuple(w[0].shape) != (256, STATE_DIM) or tuple(w[2].shape) != (256, 256) or tuple(w[4].shape) != (ACTION_DIM, 256):
        raise ValueError("plen_actor_forward implements the reference architecture 26-256-256-18 (td3.py:37-41)")
    dev = obs.device
    with torch.cuda.device(dev):
        if precision not in ("fp32", "fp16"):
            raise ValueError("precision must be 'fp32' or 'fp16'")
        fn = lib.plen_actor_forward if precision == "fp32" else lib.plen_actor_forward_tc
        rc = fn(dev.index if dev.index is not None else torch.cuda.current_device(), *[_p(t) for t in w],
                                    _p(obs), n, float(actor.max_action), float(noise_std), int(seed) & (2 ** 64 - 1), _p(out),
                                    C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    if rc != 0:
        raise RuntimeError("plen_actor_forward: %s" % lib.plen_td3_last_error().decode())
    global _tc_checked
    if precision == "fp16" and not _tc_checked:
        # once per process (it synchronises): a tensor-core launch that abandoned an mbarrier wait wrote NaN actions
        _tc_checked = True
        if lib.plen_actor_tc_timed_out() != 0:
            raise RuntimeError("plen_actor_forward_tc abandoned an mbarrier wait (tcgen05 pipeline protocol error)")
    return out


class ReplayBuffer:
    """Device ring of (state, action, next_state, reward, done) tuples -- ReplayBuffer of td3.py:122-193, batched."""

    def __init__(self, max_size=1000000, device="cuda:0", seed=0):
        if not torch.cuda.is_available():
            raise RuntimeError("the replay ring lives in HBM; there is no CPU fallback")
        self.lib = _abi.load_library()
        self.device = torch.device(device)
        self.max_size = int(max_size)
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self._rb = self.lib.plen_replay_create(self.max_size, idx)
        if not self._rb:
            raise RuntimeError("plen_replay_create: %s" % self.lib.plen_td3_last_error().decode())
        self._seed, self._draws = int(seed), 0

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def __len__(self):
        return int(self.lib.plen_replay_size(self._rb))

    @property
    def ptr(self):
        return int(self.lib.plen_replay_ptr(self._rb))

    def add(self, state, action, next_state, reward, done):
        """N tuples at once: state/next_state [N,26], action [N,18], reward [N], done [N] (bool / uint8: done_bool of
        plen_td3.py:109-110, i.e. False on TimeLimit truncation)."""
        f = lambda t, w: torch.as_tensor(t, device=self.device).float().reshape(-1, w).contiguous()
        s, a, s2 = f(state, STATE_DIM), f(action, ACTION_DIM), f(next_state, STATE_DIM)
        r = torch.as_tensor(reward, device=self.device).float().reshape(-1).contiguous()
        d = torch.as_tensor(done, device=self.device).to(torch.uint8).reshape(-1).contiguous()
        n = s.shape[0]
        if not (a.shape[0] == s2.shape[0] == r.shape[0] == d.shape[0] == n):
            raise ValueError("ReplayBuffer.add: inconsistent batch sizes")
        with torch.cuda.device(self.device):
            rc = self.lib.plen_replay_add(self._rb, _p(s), _p(a), _p(s2), _p(r), _p(d), n, self._stream())
        if rc != 0:
            raise RuntimeError("plen_replay_add: %s" % self.lib.plen_td3_last_error().decode())

    def sample(self, batch_size, return_index=False):
        """-> state, action, next_state, reward [B,1], not_done [B,1]   (td3.py:166-193)"""
        dev, b = self.device, int(batch_size)
        s = torch.empty((b, STATE_DIM), device=dev); a = torch.empty((b, ACTION_DIM), device=dev)
        s2 = torch.empty((b, STATE_DIM), device=dev); r = torch.empty((b, 1), device=dev); nd = torch.empty((b, 1), device=dev)
        idx = torch.empty(b, dtype=torch.int32, device=dev) if return_index else None
        self._draws += 1
        with torch.cuda.device(dev):
            rc = self.lib.plen_replay_sample(self._rb, b, (self._seed * 1000003 + self._draws) & (2 ** 64 - 1), _p(s), _p(a), _p(s2),
                                             _p(r), _p(nd), _p(idx), self._stream())
        if rc != 0:
            raise RuntimeError("plen_replay_sample: %s" % self.lib.plen_td3_last_error().decode())
        return (s, a, s2, r, nd, idx) if return_index else (s, a, s2, r, nd)

    def storage(self):
        """[len, 72] copy of the stored transitions in ring order (tests, checkpointing)."""
        n = len(self)
        if n == 0:
            return torch.empty((0, 72), device=self.device)
        src = self.lib.plen_replay_storage(self._rb)
        return _from_device_ptr(src, n * 72, self.device).view(n, 72).clone()

    def close(self):
        if getattr(self, "_rb", None):
            self.lib.plen_replay_destroy(self._rb)
            self._rb = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _from_device_ptr(ptr, numel, device):
    """torch float32 view of raw device memory owned by the library (no copy)."""
    class _Holder:
        pass
    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (int(numel),), "typestr": "<f4", "data": (int(ptr), False), "version": 3}
    return torch.as_tensor(h, device=device)


def _flatten_module(module):
    """Move every parameter of `module` into ONE flat float32 vector (state_dict order) and make the parameters views of it,
    so the CUDA learner (flat layouts of include/plen_b200.h) and the nn.Module / state_dict / checkpoint surface share
    the same memory."""
    ps = list(module.parameters())
    flat = torch.cat([p.detach().reshape(-1).float() for p in ps]).contiguous()
    off = 0
    for p in ps:
        n = p.numel()
        p.data = flat[off:off + n].view(p.shape)
        off += n
    return flat


class TD3Agent:                                            # td3.py:196-376
    """TD3Agent of the reference with the update rule (td3.py:259-356) running in the CUDA library (`train`): strided fp32
    GEMM kernels with fused epilogues, fused Adam, fused Polyak update -- no autograd, no cuBLAS.  `train_torch` keeps the
    same rule in plain PyTorch as the fp32 reference the tests compare against (and for CPU-only checkpoint tooling)."""

    def __init__(self, state_dim=STATE_DIM, action_dim=ACTION_DIM, max_action=1.0, discount=0.99, tau=0.005,
                 policy_noise=0.2, noise_clip=0.5, policy_freq=2, device="cuda:0", lr=3e-4, max_batch=4096, seed=0,
                 precision="fp32"):
        """precision: "fp32" = every product on the FP32 CUDA cores, within 1e-5 of torch (the parity path); "tf32" = for
        minibatches >= 512 rows, the products that fill a 128-row tile run on the tcgen05 tensor cores (3xTF32: operands
        split into two TF32 parts, FP32 accumulation; fp32-level accuracy) -- for minibatches >= 1024, where the update is
        FLOP bound.  Smaller minibatches stay on the FP32 CUDA cores in either precision."""
        if precision not in ("fp32", "tf32"):
            raise ValueError("precision must be 'fp32' or 'tf32'")
        self.precision = precision
        self.device = torch.device(device)
        self.actor = Actor(state_dim, action_dim, max_action).to(self.device)
        self.actor_target = copy.deepcopy(self.actor)
        self.critic = Critic(state_dim, action_dim).to(self.device)
        self.critic_target = copy.deepcopy(self.critic)
        self.max_action, self.discount, self.tau = max_action, discount, tau
        self.policy_noise, self.noise_clip, self.policy_freq = policy_noise, noise_clip, policy_freq
        self.lr = lr
        self.total_it = 0
        self.critic_steps = 0      # Adam step counters (torch keeps them in optimizer.state[p]["step"])
        self.actor_steps = 0
        self._draws = 0
        self._seed = int(seed)
        self._flat = {}
        self._reflatten()
        z = lambda ref: torch.zeros_like(ref)
        self._adam = {"actor_m": z(self._flat["actor"]), "actor_v": z(self._flat["actor"]),
                      "critic_m": z(self._flat["critic"]), "critic_v": z(self._flat["critic"])}
        self._grad = {"actor": z(self._flat["actor"]), "critic": z(self._flat["critic"])}
        # torch optimizers exist for the checkpoint surface (save / load of *_optimizer files) and for train_torch
        self.actor_optimizer = torch.optim.Adam(self.actor.parameters(), lr=lr)
        self.critic_optimizer = torch.optim.Adam(self.critic.parameters(), lr=lr)
        self._learner, self._max_batch = None, int(max_batch)
        self._losses = torch.zeros(2, dtype=torch.float32, device=self.device) if self.device.type == "cuda" else None

    # ---- flat storage shared with the CUDA learner
    def _reflatten(self):
        for name in ("actor", "actor_target", "critic", "critic_target"):
            self._flat[name] = _flatten_module(getattr(self, name))
        assert self._flat["actor"].numel() == _abi.TD3_ACTOR_PARAMS and self._flat["critic"].numel() == _abi.TD3_CRITIC_PARAMS

    def _cuda_handles(self):
        if self.device.type != "cuda":
            raise RuntimeError("TD3Agent.train runs in the CUDA library; there is no CPU fallback (train_torch is the test reference)")
        lib = _abi.load_library()
        if self._learner is None:
            idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
            self._learner = lib.plen_td3_create(self._max_batch, idx)
            if not self._learner:
                raise RuntimeError("plen_td3_create: %s" % lib.plen_td3_last_error().decode())
            self._hyper = _abi.PlenTd3HyperC()
            lib.plen_td3_default_hyper(C.byref(self._hyper))
            self._check(lib, lib.plen_td3_set_precision(self._learner, 1 if self.precision == "tf32" else 0))
        h = self._hyper
        h.discount, h.tau, h.policy_noise, h.noise_clip = self.discount, self.tau, self.policy_noise, self.noise_clip
        h.max_action, h.lr, h.policy_freq = self.max_action, self.lr, self.policy_freq
        P = _abi.PlenTd3ParamsC()
        for k in ("actor", "actor_target", "critic", "critic_target"):
            setattr(P, k, self._flat[k].data_ptr())
        for k in ("actor_m", "actor_v", "critic_m", "critic_v"):
            setattr(P, k, self._adam[k].data_ptr())
        P.actor_grad, P.critic_grad = self._grad["actor"].data_ptr(), self._grad["critic"].data_ptr()
        return lib, P, h

    def _idx(self):
        return self.device.index if self.device.index is not None else torch.cuda.current_device()

    def select_action(self, state, expl_noise=0.0, precision="fp32"):
        """Batched: state [N,26] on the device -> action [N,18]; expl_noise = plen_td3.py:101-104 (std = max_action * expl_noise)."""
        self._draws += 1
        # the noise stream is keyed by the agent's seed as well as the draw counter: data-parallel ranks (one agent per GPU,
        # seeded per rank) must not explore with identical noise rows
        return actor_forward(self.actor, torch.as_tensor(state, device=self.device).reshape(-1, STATE_DIM),
                             noise_std=self.max_action * expl_noise, seed=(self._seed * 1000003 + self._draws) & (2 ** 64 - 1),
                             precision=precision)

    def train(self, replay_buffer, batch_size=100, batch=None, noise=None, return_losses=False, grad_hook=None):
        """One TD3 update (td3.py:259-356) in the CUDA library.

        replay_buffer: the device ReplayBuffer (sampled inside the library); or pass an explicit minibatch
        batch = (state, action, next_state, reward, not_done) -- used by the parity tests together with `noise`
        ([B,18] standard-normal samples for the target policy smoothing).  grad_hook(flat_grad) runs between the
        gradient kernels and Adam: a data-parallel learner all-reduces there (NCCL, SURVEY.md 8e).
        Returns (actor_loss, critic_loss) device scalars when return_losses (actor_loss is None off the policy step)."""
        lib, P, h = self._cuda_handles()
        self.total_it += 1
        self._draws += 1
        seed = (self._seed * 1000003 + self._draws) & (2 ** 64 - 1)
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        policy = self.total_it % self.policy_freq == 0
        with torch.cuda.device(self.device):
            if batch is not None:
                s, a, s2, r, nd = [torch.as_tensor(x, device=self.device).float().contiguous() for x in batch]
                rc = lib.plen_td3_set_batch(self._learner, _p(s), _p(a), _p(s2), _p(r.reshape(-1)), _p(nd.reshape(-1)), s.shape[0], st)
                self._check(lib, rc)
            if batch is None and noise is None and grad_hook is None:
                # the whole step in one library call
                self.critic_steps += 1
                if policy:
                    self.actor_steps += 1
                rc = lib.plen_td3_train(self._learner, C.byref(P), C.byref(h), replay_buffer._rb, int(batch_size), self.total_it,
                                        self.critic_steps, max(1, self.actor_steps), seed, _p(self._losses), st)
                self._check(lib, rc)
            else:
                if batch is None:
                    self._check(lib, lib.plen_td3_sample(self._learner, replay_buffer._rb, int(batch_size), seed ^ 0x9E3779B97F4A7C15, st))
                nz = None if noise is None else torch.as_tensor(noise, device=self.device).float().contiguous()
                self._check(lib, lib.plen_td3_critic_grads(self._learner, C.byref(P), C.byref(h), _p(nz), seed,
                                                           C.c_void_p(self._losses.data_ptr() + 4), st))
                if grad_hook is not None:
                    grad_hook(self._grad["critic"])
                self.critic_steps += 1
                self._check(lib, lib.plen_td3_adam(P.critic, P.critic_grad, P.critic_m, P.critic_v, _abi.TD3_CRITIC_PARAMS,
                                                   self.critic_steps, C.byref(h), self._idx(), st))
                if policy:
                    self._check(lib, lib.plen_td3_actor_grads(self._learner, C.byref(P), C.byref(h), _p(self._losses), st))
                    if grad_hook is not None:
                        grad_hook(self._grad["actor"])
                    self.actor_steps += 1
                    self._check(lib, lib.plen_td3_adam(P.actor, P.actor_grad, P.actor_m, P.actor_v, _abi.TD3_ACTOR_PARAMS,
                                                       self.actor_steps, C.byref(h), self._idx(), st))
                    self._check(lib, lib.plen_td3_soft_update(P.critic_target, P.critic, _abi.TD3_CRITIC_PARAMS, float(self.tau), self._idx(), st))
                    self._check(lib, lib.plen_td3_soft_update(P.actor_target, P.actor, _abi.TD3_ACTOR_PARAMS, float(self.tau), self._idx(), st))
        if return_losses:
            return (self._losses[0].clone() if policy else None), self._losses[1].clone()
        return None

    @staticmethod
    def _check(lib, rc):
        if rc != 0:
            raise RuntimeError("libplen_b200 TD3 learner: %s" % lib.plen_td3_last_error().decode())

    def kernel_launches(self):
        return int(_abi.load_library().plen_td3_launches(self._learner)) if self._learner else 0

    def train_torch(self, batch, noise=None):
        """The same update in plain PyTorch (autograd + torch.optim.Adam): the fp32 reference of the tests.  batch =
        (state, action, next_state, reward [B,1], not_done [B,1]); noise [B,18] standard normal (None: torch.randn)."""
        self.total_it += 1
        state, action, next_state, reward, not_done = batch
        with torch.no_grad():
            nz = torch.randn_like(action) if noise is None else noise
            nz = (nz * self.policy_noise).clamp(-self.noise_clip, self.noise_clip)
            next_action = (self.actor_target(next_state) + nz).clamp(-self.max_action, self.max_action)
            target_Q1, target_Q2 = self.critic_target(next_state, next_action)
            target_Q = reward + not_done * self.discount * torch.min(target_Q1, target_Q2)
        current_Q1, current_Q2 = self.critic(state, action)
        critic_loss = F.mse_loss(current_Q1, target_Q) + F.mse_loss(current_Q2, target_Q)
        self.critic_optimizer.zero_grad()
        critic_loss.backward()
        self.critic_optimizer.step()
        actor_loss = None
        if self.total_it % self.policy_freq == 0:
            actor_loss = -self.critic.Q1(state, self.actor(state)).mean()
            self.actor_optimizer.zero_grad()
            actor_loss.backward()
            self.actor_optimizer.step()
            with torch.no_grad():
                for param, target_param in zip(self.critic.parameters(), self.critic_target.parameters()):
                    target_param.copy_(self.tau * param + (1 - self.tau) * target_param)
                for param, target_param in zip(self.actor.parameters(), self.actor_target.parameters()):
                    target_param.copy_(self.tau * param + (1 - self.tau) * target_param)
        return actor_loss, critic_loss

    # ---- checkpoints: same four files and formats as td3.py:358-376
    def _sync_optimizer_state(self, opt, module, m, v, steps):
        off = 0
        for p in module.parameters():
            n = p.numel()
            opt.state[p] = {"step": torch.tensor(float(steps)), "exp_avg": m[off:off + n].view(p.shape).clone(),
                            "exp_avg_sq": v[off:off + n].view(p.shape).clone()}
            off += n

    def _load_optimizer_state(self, opt, module, m, v):
        off, steps = 0, 0
        for p in module.parameters():
            n = p.numel()
            st = opt.state.get(p, {})
            if "exp_avg" in st:
                m[off:off + n].copy_(st["exp_avg"].reshape(-1))
                v[off:off + n].copy_(st["exp_avg_sq"].reshape(-1))
                steps = int(float(st["step"]))
            off += n
        return steps

    def save(self, filename):
        self._sync_optimizer_state(self.critic_optimizer, self.critic, self._adam["critic_m"], self._adam["critic_v"], self.critic_steps)
        self._sync_optimizer_state(self.actor_optimizer, self.actor, self._adam["actor_m"], self._adam["actor_v"], self.actor_steps)
        torch.save(self.critic.state_dict(), filename + "_critic")
        torch.save(self.critic_optimizer.state_dict(), filename + "_critic_optimizer")
        torch.save(self.actor.state_dict(), filename + "_actor")
        torch.save(self.actor_optimizer.state_dict(), filename + "_actor_optimizer")

    def load(self, filename, optimizers=True, sync_targets=False):
        """TD3Agent.load (td3.py:366-376).  Like the reference, the TARGET networks are left untouched (there they keep
        whatever they held before the call); sync_targets=True copies the loaded weights into them, which is what one wants
        before continuing training from a checkpoint.  The reference's optimizer files are python-2 era pickles and need
        weights_only=False -- only load optimizer files you trust, or pass optimizers=False (inference needs none)."""
        # load_state_dict copies in place, so the parameters stay views of the flat vectors
        self.critic.load_state_dict(torch.load(filename + "_critic", map_location=self.device))
        self.actor.load_state_dict(torch.load(filename + "_actor", map_location=self.device))
        if optimizers:   # the reference's optimizer files are python-2 pickles that need weights_only=False (SURVEY.md 4)
            self.critic_optimizer.load_state_dict(torch.load(filename + "_critic_optimizer", map_location=self.device, weights_only=False))
            self.actor_optimizer.load_state_dict(torch.load(filename + "_actor_optimizer", map_location=self.device, weights_only=False))
            self.critic_steps = self._load_optimizer_state(self.critic_optimizer, self.critic, self._adam["critic_m"], self._adam["critic_v"])
            self.actor_steps = self._load_optimizer_state(self.actor_optimizer, self.actor, self._adam["actor_m"], self._adam["actor_v"])
        if sync_targets:
            self._flat["actor_target"].copy_(self._flat["actor"])
            self._flat["critic_target"].copy_(self._flat["critic"])

    def close(self):
        if getattr(self, "_learner", None):
            _abi.load_library().plen_td3_destroy(self._learner)
            self._learner = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
