"""TEST-ONLY float64 references for the TD3 kernels of libplen_b200.so: the counter-based noise generators, the replay draw of
the one-call update, an FP16 rounding model of the tensor-core actor and a float64 twin of the TD3 update rule."""
import copy

import numpy as np
import torch
import torch.nn.functional as F

M64 = (1 << 64) - 1
FNV = 0x100000001B3                 # counter multiplier of every generator
U32_SCALE = np.float32(2.3283064e-10)


def mix32(x):
    """splitmix64 finaliser, upper 32 bits (mix32 / hash32 / mixh of the CUDA sources); x: uint64 array."""
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return ((x ^ (x >> np.uint64(31))) >> np.uint64(32)).astype(np.uint32)


def _box_muller(ctr, xor):
    """standard normal draw of counter ctr: u1 = (h + 1) 2^-32, u2 = h' 2^-32 in float32 as the kernels form them, then
    sqrt(-2 ln u1) cos(2 pi u2) in float64"""
    u1 = (mix32(ctr).astype(np.float32) + np.float32(1.0)) * U32_SCALE
    with np.errstate(over="ignore"):
        u2 = mix32(ctr ^ np.uint64(xor)).astype(np.float32) * U32_SCALE
    u1, u2 = u1.astype(np.float64), u2.astype(np.float64)
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def _counters(seed, rows, cols, row_stride):
    m = np.arange(rows, dtype=np.uint64)[:, None]
    n = np.arange(cols, dtype=np.uint64)[None, :]
    with np.errstate(over="ignore"):
        return np.uint64((int(seed) * FNV) & M64) + m * np.uint64(row_stride) + n


def learner_noise(seed, rows, cols=18):
    """[rows, cols] policy-smoothing noise of the learner's EPI_BIAS_TANH_NOISE epilogue when no noise buffer is given
    (plen_td3_learn.cu): counter seed * FNV + 64 m + n."""
    return _box_muller(_counters(seed, rows, cols, 64), 0x5DEECE66D1234567)


def actor_noise(seed, rows, cols=18):
    """[rows, cols] standard-normal exploration draws of plen_actor_forward / plen_actor_forward_tc: counter
    seed * FNV + 32 row + joint."""
    return _box_muller(_counters(seed, rows, cols, 32), 0xA5A5A5A5DEADBEEF)


def train_seed(agent):
    """seed TD3Agent.train passed to the library on its last call"""
    return (agent._seed * 1000003 + agent._draws) & M64


def graph_draw_seed(s):
    """seed of plen_replay_sample that draws the rows k_sample_sa draws in plen_td3_train for call seed s"""
    return (s * 2654435761 + 1) & M64


def replay_rows(rb, batch, seed):
    """(state, action, next_state, reward [B,1], not_done [B,1], index) of plen_replay_sample(seed) on ReplayBuffer rb"""
    import ctypes as C
    dev = rb.device
    s = torch.empty((batch, 26), device=dev); a = torch.empty((batch, 18), device=dev); s2 = torch.empty((batch, 26), device=dev)
    r = torch.empty((batch, 1), device=dev); nd = torch.empty((batch, 1), device=dev)
    idx = torch.empty(batch, dtype=torch.int32, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    with torch.cuda.device(dev):
        rc = rb.lib.plen_replay_sample(rb._rb, batch, seed, p(s), p(a), p(s2), p(r), p(nd), p(idx),
                                       C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    assert rc == 0, rb.lib.plen_td3_last_error().decode()
    return s, a, s2, r, nd, idx


# ---- FP16 tensor-core actor (plen_actor_tc.cu): fp16 operands (round to nearest, saturating), exact accumulation
def f16(x):
    """x (float64 tensor) -> the float64 value of its saturating round-to-nearest FP16 (pack_f16)"""
    return x.clamp(-65504.0, 65504.0).to(torch.float32).to(torch.float16).to(torch.float64)


def actor_fp16_model(actor, obs, max_action=None):
    """float64 output of plen_actor_forward_tc for obs [N,26]: observations and weights rounded to FP16, each hidden layer
    relu(acc + b) rounded to FP16, output max_action tanh(acc3 + b3); the products themselves exact."""
    d = lambda t: t.detach().to(torch.float64)
    ma = actor.max_action if max_action is None else max_action
    h = f16(d(obs))
    h = f16(torch.relu(h @ f16(d(actor.fc1.weight)).T + d(actor.fc1.bias)))
    h = f16(torch.relu(h @ f16(d(actor.fc2.weight)).T + d(actor.fc2.bias)))
    return ma * torch.tanh(h @ f16(d(actor.fc3.weight)).T + d(actor.fc3.bias))


# ---- TD3 update rule (td3.py:259-356) in float64
class Td3Twin:
    """float64 copy of a TD3Agent's four networks and Adam states, stepped by the reference rule with autograd and
    torch.optim.Adam; the minibatch and the standard-normal smoothing noise are given."""

    def __init__(self, agent):
        self.actor = copy.deepcopy(agent.actor).double()
        self.actor_target = copy.deepcopy(agent.actor_target).double()
        self.critic = copy.deepcopy(agent.critic).double()
        self.critic_target = copy.deepcopy(agent.critic_target).double()
        self.max_action, self.discount, self.tau = agent.max_action, agent.discount, agent.tau
        self.policy_noise, self.noise_clip, self.policy_freq = agent.policy_noise, agent.noise_clip, agent.policy_freq
        self.total_it = agent.total_it
        self.actor_optimizer = torch.optim.Adam(self.actor.parameters(), lr=agent.lr)
        self.critic_optimizer = torch.optim.Adam(self.critic.parameters(), lr=agent.lr)
        for opt, module, m, v, steps in ((self.critic_optimizer, self.critic, agent._adam["critic_m"], agent._adam["critic_v"], agent.critic_steps),
                                         (self.actor_optimizer, self.actor, agent._adam["actor_m"], agent._adam["actor_v"], agent.actor_steps)):
            if steps == 0:
                continue
            off = 0
            for p in module.parameters():
                n = p.numel()
                opt.state[p] = {"step": torch.tensor(float(steps)),
                                "exp_avg": m[off:off + n].view(p.shape).to(torch.float64).clone(),
                                "exp_avg_sq": v[off:off + n].view(p.shape).to(torch.float64).clone()}
                off += n
        self._rms = {}
        for name in ("actor", "critic"):
            self._track(name)

    def _track(self, name):
        """smallest bias-corrected RMS gradient sqrt(v_hat) seen so far, per parameter (inf before the first step)"""
        opt, module = getattr(self, name + "_optimizer"), getattr(self, name)
        if not opt.state:
            self._rms[name] = torch.full_like(self.flat(name), float("inf"))
            return
        b2 = opt.param_groups[0]["betas"][1]
        r = torch.cat([(opt.state[p]["exp_avg_sq"] / (1 - b2 ** float(opt.state[p]["step"]))).sqrt().reshape(-1)
                       for p in module.parameters()])
        self._rms[name] = torch.minimum(self._rms[name], r) if name in self._rms else r

    def adam_sensitive(self, name, rel=1e-2):
        """parameters whose Adam step has been ill-conditioned: sqrt(v_hat) fell below `rel` times the network's RMS of it at
        some update.  There m_hat / (sqrt(v_hat) + eps) turns a gradient difference at the level of fp32 rounding into a
        step difference of up to 2 lr, whichever arithmetic (summation order, split-K atomics) produced the gradient."""
        r = self._rms[name]
        fin = r[torch.isfinite(r)]
        if fin.numel() == 0:
            return torch.zeros_like(r, dtype=torch.bool)
        return r < rel * fin.square().mean().sqrt()

    def flat(self, name):
        return torch.cat([p.detach().reshape(-1) for p in getattr(self, name).parameters()])

    def moments(self, name):
        opt, module = getattr(self, name + "_optimizer"), getattr(self, name)
        return (torch.cat([opt.state[p]["exp_avg"].reshape(-1) for p in module.parameters()]),
                torch.cat([opt.state[p]["exp_avg_sq"].reshape(-1) for p in module.parameters()]))

    def update(self, batch, noise):
        """one update; batch = (s, a, s', r [B,1], not_done [B,1]), noise [B,18] standard normal.  -> (actor_loss or None,
        critic_loss) as floats"""
        self.total_it += 1
        state, action, next_state, reward, not_done = [torch.as_tensor(x).to(torch.float64) for x in batch]
        noise = torch.as_tensor(noise).to(device=state.device, dtype=torch.float64)
        with torch.no_grad():
            nz = (noise * self.policy_noise).clamp(-self.noise_clip, self.noise_clip)
            next_action = (self.actor_target(next_state) + nz).clamp(-self.max_action, self.max_action)
            tq1, tq2 = self.critic_target(next_state, next_action)
            target_q = reward + not_done * self.discount * torch.min(tq1, tq2)
        q1, q2 = self.critic(state, action)
        critic_loss = F.mse_loss(q1, target_q) + F.mse_loss(q2, target_q)
        self.critic_optimizer.zero_grad()
        critic_loss.backward()
        self.critic_optimizer.step()
        self._track("critic")
        actor_loss = None
        if self.total_it % self.policy_freq == 0:
            actor_loss = -self.critic.Q1(state, self.actor(state)).mean()
            self.actor_optimizer.zero_grad()
            actor_loss.backward()
            self.actor_optimizer.step()
            self._track("actor")
            with torch.no_grad():
                for net, tgt in ((self.critic, self.critic_target), (self.actor, self.actor_target)):
                    for p, tp in zip(net.parameters(), tgt.parameters()):
                        tp.copy_(self.tau * p + (1 - self.tau) * tp)
            actor_loss = actor_loss.item()
        return actor_loss, critic_loss.item()
