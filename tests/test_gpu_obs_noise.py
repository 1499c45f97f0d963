"""Per-robot observation noise (plen_set_env_obs_noise, PlenVecEnv.set_obs_noise) on the GPU: an all-zero table is the stock
path bit for bit, noise never feeds back into reward, done or the physics, the draws match the numpy twin (tests/obs_noise_util.py)
and have the stated statistics, the bias is drawn at every reset path and nowhere else, results depend neither on batch
layout nor on the step path, a captured CUDA graph draws new noise per replay, snapshots continue a noisy run, and bad
arguments are refused."""
import ctypes as C
import os

import numpy as np
import pytest

import obs_noise_util as U

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

PLEN_E_ARG, PLEN_E_STATE = -1, -3
# device Gaussians (sqrtf / logf / cospif in float32) against the twin's float64 Box-Muller of the same float32 uniforms: measured
# worst 1.18e-7 (1 + |n|) over 4.8 million draws on a B200 at 1000 W (test_device_gaussians_against_the_twin); held to 3x that
GPU_NORMAL_REL = 3.5e-7
F32_EPS = 2.0 ** -23
SEED = 20261022


def _mk(n, **kw):
    from plen_ml_walk_b200.vec_env import PlenVecEnv
    return PlenVecEnv(n, device="cuda:0", **kw)


def _bits(t):
    return t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t


def _eq(a, b):
    """bit for bit (NaN payloads and the sign of zero included)"""
    return a.shape == b.shape and bool(torch.equal(_bits(a), _bits(b)))


def _acts(n, steps, seed, amp=1.0):
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    return [torch.empty((n, 18), device="cuda").uniform_(-amp, amp, generator=g) for _ in range(steps)]


def _noise(n, seed=5):
    """per-robot, per-word parameters with every 5th word off"""
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    s = torch.empty((n, 24), device="cuda").uniform_(0.0, 0.05, generator=g)
    b = torch.empty((n, 24), device="cuda").uniform_(0.0, 0.05, generator=g)
    s[:, ::5] = 0.0
    b[:, ::5] = 0.0
    p = torch.empty(n, device="cuda").uniform_(0.0, 0.2, generator=g)
    return s, b, p


def _step(env, a):
    obs, rew, done, info = env.step(a)
    out = [obs.clone(), rew.clone(), done.clone(), info["timeout"].clone(),
           torch.where(done[:, None], info["terminal_obs"], torch.zeros_like(obs))]
    if "clean_obs" in info:
        out += [info["clean_obs"].clone(), torch.where(done[:, None], info["clean_terminal_obs"], torch.zeros_like(obs))]
    return out


def _np(t):
    return t.detach().cpu().numpy()


def test_zero_noise_is_stock():
    """a table with all-zero sigma, bias std and flip probability: obs, reward, done, timeout, terminal_obs and records equal a
    context that never called the setter, bit for bit, over 50 steps of 4,096 robots with auto-resets"""
    n = 4096
    a, b = _mk(n), _mk(n)
    b.set_obs_noise(0.0, 0.0, 0.0, seed=SEED)
    assert _eq(a.reset(), b.reset())
    resets = 0
    for x in _acts(n, 50, 1):
        sa, sb = _step(a, x), _step(b, x)
        for u, v in zip(sa, sb):
            assert _eq(u, v)
        resets += int(sa[2].sum())
    assert resets > 100
    assert _eq(a.debug_records(), b.debug_records())


def test_noise_does_not_feed_back():
    """with noise on, the clean observations, rewards, done flags, timeouts, clean terminal observations and records equal a
    stock context bit for bit; the noisy observations do differ"""
    n = 4096
    a, b = _mk(n), _mk(n)
    b.set_obs_noise(*_noise(n), seed=SEED)
    a.reset(); b.reset()
    for x in _acts(n, 40, 2):
        sa, sb = _step(a, x), _step(b, x)
        assert _eq(sa[0], sb[5]) and _eq(sa[4], sb[6])
        for k in (1, 2, 3):
            assert _eq(sa[k], sb[k])
        assert not _eq(sa[0], sb[0])
    assert _eq(a.debug_records(), b.debug_records())


def _check_words(got, clean, sigma, bias, p, gid, ctr, stream):
    exp, _ = U.apply(clean, sigma, bias, p, SEED, gid, ctr, stream)
    z = np.abs(U.normal(U.key(SEED, gid[:, None], ctr.astype(np.uint64)[:, None], stream, np.arange(24)[None, :])))
    err = np.abs(got[:, :24] - exp[:, :24])
    round_ = 2 * F32_EPS * (np.abs(clean[:, :24]) + sigma * z + np.abs(bias))
    assert (err <= sigma * GPU_NORMAL_REL * (1 + z) + round_).all()
    assert (got[:, 24:] == exp[:, 24:]).all()


def test_draws_match_the_twin_and_bias_follows_resets():
    """step after step: obs = clean + b + sigma n (stream 0) for running robots, terminal_obs with the finished episode's bias,
    the new bias beta n' (stream 2) and the reset observation (streams 3 / 4) for auto-reset robots; flips and counters exact.
    The bias stays constant within an episode and is redrawn by auto-resets, by explicit resets of the masked robots only and
    by the numeric guard's forced reset."""
    n, first = 3000, 777
    env = _mk(n)
    s, b, p = _noise(n)
    env.set_obs_noise(s, b, p, seed=SEED, first_env_id=first)
    gid = first + np.arange(n)
    sig, beta, pp = _np(s), _np(b), _np(p)
    obs0 = _np(env.reset())
    nz = env.get_obs_noise()
    assert (_np(nz["counter"]).view(np.uint32) == 1).all()
    _check_words(obs0, _np(env.clean_obs()[0]), sig, _np(nz["bias"]), pp, gid, np.zeros(n, np.uint32), U.NS_ROBS)
    nb = U.new_bias(beta, SEED, gid, np.zeros(n, np.uint32))
    assert (np.abs(_np(nz["bias"]) - nb) <= beta * GPU_NORMAL_REL * (1 + np.abs(nb) / np.maximum(beta, 1e-30)) + F32_EPS * np.abs(nb)).all()
    acts = _acts(n, 30, 3)
    for t, x in enumerate(acts):
        before = env.get_obs_noise()
        b0, c0 = _np(before["bias"]), _np(before["counter"]).view(np.uint32)
        if t == 10:         # the numeric guard: a non-finite base position retires robots 0..9 with a forced reset
            qpos, qvel, aux = env.get_state()
            qpos[:10, 0] = float("nan")
            env.set_state(qpos, qvel, aux)
        obs, rew, done, info = env.step(x)
        co, ct = (_np(v) for v in env.clean_obs())
        o, d, tobs = _np(obs), _np(done), _np(info["terminal_obs"])
        after = env.get_obs_noise()
        b1, c1 = _np(after["bias"]), _np(after["counter"]).view(np.uint32)
        assert (c1 == c0 + 1).all()
        run = ~d
        _check_words(o[run], co[run], sig[run], b0[run], pp[run], gid[run], c0[run], U.NS_OBS)
        assert _eq(torch.from_numpy(b1[run]), torch.from_numpy(b0[run]))
        if d.any():
            _check_words(tobs[d], ct[d], sig[d], b0[d], pp[d], gid[d], c0[d], U.NS_OBS)
            nb = U.new_bias(beta[d], SEED, gid[d], c0[d])
            tol = beta[d] * GPU_NORMAL_REL * (1 + np.abs(nb) / np.maximum(beta[d], 1e-30)) + F32_EPS * np.abs(nb)
            assert (np.abs(b1[d] - nb) <= tol).all()
            _check_words(o[d], co[d], sig[d], b1[d], pp[d], gid[d], c0[d], U.NS_ROBS)
        if t == 10:
            assert d[:10].all()
    # explicit reset of every third robot: only those redraw
    mask = np.arange(n) % 3 == 0
    before = env.get_obs_noise()
    b0, c0 = _np(before["bias"]), _np(before["counter"]).view(np.uint32)
    o_prev = env._obs.clone()
    env.reset(torch.from_numpy(mask).cuda())
    after = env.get_obs_noise()
    b1, c1 = _np(after["bias"]), _np(after["counter"]).view(np.uint32)
    assert (c1 == c0 + mask).all()
    assert (b1[~mask] == b0[~mask]).all() and not (b1[mask] == b0[mask]).all()
    assert _eq(env._obs[torch.from_numpy(~mask).cuda()], o_prev[torch.from_numpy(~mask).cuda()])
    co = _np(env.clean_obs()[0])
    _check_words(_np(env._obs)[mask], co[mask], sig[mask], b1[mask], pp[mask], gid[mask], c0[mask], U.NS_ROBS)


def test_device_gaussians_against_the_twin():
    """bias_std = 1 makes each new episode's bias the device's Gaussian itself (beta n' with beta = 1 is exact): 40,000 robots x
    24 words x 5 explicit resets against the twin's float64 Box-Muller of the same uniforms, within GPU_NORMAL_REL (1 + |n|)"""
    n = 40000
    env = _mk(n)
    env.set_obs_noise(0.0, 1.0, 0.0, seed=SEED, first_env_id=3)
    gid = 3 + np.arange(n)
    worst = 0.0
    for r in range(5):
        env.reset()
        got = _np(env.get_obs_noise()["bias"]).astype(np.float64)
        ref = U.new_bias(np.ones((n, 24), np.float32), SEED, gid, np.full(n, r, np.uint32))
        err = np.abs(got - ref) / (1 + np.abs(ref))
        worst = max(worst, float(err.max()))
    print("device Gaussians vs twin: worst %.2e (1 + |n|) over %d draws" % (worst, 5 * n * 24))
    assert worst <= GPU_NORMAL_REL


def test_statistics():
    """sigma = 1 on every word of 40,000 robots over 30 steps (28.8 million draws, no bias): the mean and variance of
    noisy - clean within 5 standard errors of 0 and 1, correlations between neighbouring words and consecutive steps below
    5 / sqrt(n), flips at p = 0.3 within 5 standard errors"""
    n, steps = 40000, 30
    env = _mk(n)
    env.set_obs_noise(1.0, 0.0, 0.3, seed=SEED)
    env.reset()
    diffs, flips = [], []
    for x in _acts(n, steps, 4, amp=0.2):
        obs, _, _, info = env.step(x)
        co = info["clean_obs"]
        diffs.append((obs[:, :24].double() - co[:, :24].double()).cpu())
        flips.append((obs[:, 24:] != co[:, 24:]).double().cpu())
    d = torch.stack(diffs)             # [steps, n, 24]
    m = d.numel()
    assert abs(float(d.mean())) < 5 / m ** 0.5
    assert abs(float(d.var()) - 1.0) < 5 * (2.0 / m) ** 0.5
    def corr(x, y):
        x, y = x.flatten() - x.mean(), y.flatten() - y.mean()
        return float((x * y).sum() / (x.norm() * y.norm()))
    k = d[:, :, :-1].numel()
    assert abs(corr(d[:, :, :-1], d[:, :, 1:])) < 5 / k ** 0.5
    k = d[:-1].numel()
    assert abs(corr(d[:-1], d[1:])) < 5 / k ** 0.5
    f = torch.stack(flips)
    assert abs(float(f.mean()) - 0.3) < 5 * (0.21 / f.numel()) ** 0.5


def test_layout_independence():
    """two contexts [0, k) and [k, n) with first_env_id 0 and k equal one context of n; step equals step_host; the first m
    robots are the same at n = 1, 37, 2,085 and 40,000"""
    sizes = (1, 37, 2085, 40000)
    n, k = sizes[-1], 13000
    acts = _acts(n, 12, 6)
    s, b, p = _noise(n)

    def run(env, lo, hi):
        env.set_obs_noise(s[lo:hi], b[lo:hi], p[lo:hi], seed=SEED, first_env_id=lo)
        out = [env.reset().clone()]
        for x in acts:
            out.append(_step(env, x[lo:hi].contiguous())[0])
        return torch.stack(out)

    big = run(_mk(n), 0, n)
    assert _eq(torch.cat([run(_mk(k), 0, k), run(_mk(n - k), k, n)], 1), big)
    for m in sizes[:-1]:
        assert _eq(run(_mk(m), 0, m), big[:, :m])
    # step_host against step, auto-reset on, same noise
    m = 20000
    a, h = _mk(m), _mk(m)
    for e in (a, h):
        e.set_obs_noise(s[:m], b[:m], p[:m], seed=SEED)
        e.reset()
    ob = torch.empty((m, 26)).pin_memory(); rw = torch.empty(m).pin_memory()
    dn = torch.empty(m, dtype=torch.uint8).pin_memory(); to = torch.empty(m, dtype=torch.uint8).pin_memory()
    for x in acts:
        oa, ra, da, ta, _ = _step(a, x[:m].contiguous())[:5]
        h.step_host(x[:m].cpu().pin_memory(), ob, rw, dn, to)
        assert _eq(oa.cpu(), ob) and _eq(ra.cpu(), rw) and _eq(da.cpu(), dn.bool()) and _eq(ta.cpu(), to.bool())
        assert _eq(a.clean_obs()[0], h.clean_obs()[0])


@pytest.mark.parametrize("n", [1024, 4096])
def test_cuda_graph_replays_draw_new_noise(n):
    """a captured step: 20 replays equal 20 direct calls bit for bit (obs, reward, done, terminal_obs and the clean words), and
    consecutive replays draw different noise"""
    acts = _acts(n, 20, 7)
    a, b = _mk(n), _mk(n)
    for e in (a, b):
        e.set_obs_noise(*_noise(n), seed=SEED)
        e.reset()
    direct = [_step(a, x) for x in acts]
    static_act = acts[0].clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            out = b.step(static_act)
    torch.cuda.current_stream().wait_stream(side)
    prev = None
    for k, x in enumerate(acts):
        static_act.copy_(x)
        graph.replay()
        obs, rew, done, info = out
        got = [obs, rew, done, info["timeout"], torch.where(done[:, None], info["terminal_obs"], torch.zeros_like(obs)),
               info["clean_obs"], torch.where(done[:, None], info["clean_terminal_obs"], torch.zeros_like(obs))]
        for u, v in zip(direct[k], got):
            assert _eq(u, v), "replay %d" % k
        if prev is not None:
            assert not _eq(obs - info["clean_obs"], prev)
        prev = (obs - info["clean_obs"]).clone()


def test_snapshots_continue_and_clear_restores_stock(tmp_path):
    """save_state / load_state continue a noisy run bit for bit; clear_obs_noise makes the context the stock path again"""
    n = 4096
    acts = _acts(n, 20, 8)
    a = _mk(n)
    a.set_obs_noise(*_noise(n), seed=SEED, first_env_id=5)
    a.reset()
    for x in acts[:10]:
        a.step(x)
    path = str(tmp_path / "noisy.pt")
    a.save_state(path)
    ref = [_step(a, x) for x in acts[10:]]
    b = _mk(n)
    b.load_state(path)
    nz = b.get_obs_noise()
    assert nz["active"] and nz["seed"] == SEED and nz["first_env_id"] == 5
    for k, x in enumerate(acts[10:]):
        for u, v in zip(ref[k], _step(b, x)):
            assert _eq(u, v)
    # a snapshot without noise clears it
    stock = _mk(n)
    stock.reset()
    p2 = str(tmp_path / "stock.pt")
    stock.save_state(p2)
    b.load_state(p2)
    assert not b.get_obs_noise()["active"]
    for x in acts[:10]:
        sa, sb = _step(stock, x), _step(b, x)
        assert len(sb) == 5
        for u, v in zip(sa, sb):
            assert _eq(u, v)
    # clear_obs_noise on a running noisy context
    c = _mk(n)
    c.load_state(path)
    c.clear_obs_noise()
    d = _mk(n)
    d.load_state(path)
    d.clear_obs_noise()
    for x in acts[10:]:
        sc, ss = _step(c, x), _step(d, x)
        for u, v in zip(sc, ss):
            assert _eq(u, v)
    assert _eq(c.debug_records(), a.debug_records())


def test_validation_and_launch_counts():
    """ValueError on bad shapes and values, PLEN_E_ARG for a negative first_env_id at the C level, PLEN_E_STATE for the state
    setter and the clean observations without a table; a step still launches 13 kernels per range and a reset one"""
    n = 64
    env = _mk(n)
    lib = env.lib
    with pytest.raises(RuntimeError):
        env.clean_obs()
    assert lib.plen_get_clean_obs(env._ctx, env._p(env._obs), None, None) == PLEN_E_STATE
    assert lib.plen_set_env_obs_noise_state(env._ctx, None, None, None) == PLEN_E_STATE
    assert lib.plen_set_env_obs_noise(env._ctx, None, None, None, C.c_ulonglong(1), C.c_longlong(-1), None) == PLEN_E_ARG
    assert not env.get_obs_noise()["active"]
    for bad in (dict(std=-0.1), dict(std=float("nan")), dict(std=torch.zeros(n, 23)), dict(bias_std=float("inf")),
                dict(bias_std=torch.zeros(3)), dict(contact_flip=1.5), dict(contact_flip=-0.1), dict(contact_flip=torch.zeros(n, 2)),
                dict(first_env_id=-3), dict(seed=-1)):
        with pytest.raises(ValueError):
            env.set_obs_noise(**bad)
    assert not env.get_obs_noise()["active"]
    env.set_obs_noise(torch.full((24,), 0.01), torch.full((n,), 0.02), 0.1, seed=3)
    nz = env.get_obs_noise()
    assert nz["active"] and (nz["std"] == 0.01).all() and (nz["bias_std"] == 0.02).all()
    assert torch.allclose(nz["contact_flip"], torch.full((n,), 0.1, device="cuda"))
    env.set_obs_noise(contact_flip=0.0)
    assert (env.get_obs_noise()["std"] == 0.01).all() and env.get_obs_noise()["seed"] == 3
    x = _acts(n, 1, 9)[0]
    l0 = env.launches
    env.step(x)
    assert env.launches - l0 == 13
    env.reset()
    assert env.launches - l0 == 14
    env.clear_obs_noise()
    assert not env.get_obs_noise()["active"]
    assert lib.plen_get_clean_obs(env._ctx, env._p(env._obs), None, None) == PLEN_E_STATE
