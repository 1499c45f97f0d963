"""Per-robot servo command latency (plen_set_env_latency / PlenVecEnv.set_env_latency, SURVEY.md 8f-3) on the GPU: zero delays
are the stock path bit for bit, delayed steps are the stock ticks driven with the scheduled targets (tests/latency_util.py),
resets forget the history, delays may change every step, the result depends neither on batch position nor on the step path,
snapshots continue a run bit for bit, and tick() ignores the latency."""
import numpy as np
import pytest

from latency_util import CommandSchedule

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _mk(n, **kw):
    from plen_ml_walk_b200.vec_env import PlenVecEnv
    return PlenVecEnv(n, device="cuda:0", **kw)


def _same(a, b):
    return bool(torch.equal(a, b) or torch.equal(torch.nan_to_num(a.float(), nan=1234.5), torch.nan_to_num(b.float(), nan=1234.5)))


def _acts(n, steps, seed, amp=1.0):
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    return [torch.empty((n, 18), device="cuda").uniform_(-amp, amp, generator=g) for _ in range(steps)]


def _delays(n, seed, hi=8):
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    return torch.randint(0, hi + 1, (n,), device="cuda", generator=g, dtype=torch.int32)


def _physics(env):
    qpos, qvel, aux = env.get_state()
    return qpos.clone(), qvel.clone(), aux[:, :8].clone()


def test_zero_delays_are_bit_identical_to_the_stock_path():
    """Delay 0 with the history allocated: 4,096 robots, 50 agent-space steps with auto-reset, obs / reward / done and the state
    records equal to a context that never called the setter."""
    n = 4096
    stock, lat = _mk(n), _mk(n)
    lat.set_env_latency(0)
    stock.reset(); lat.reset()
    dones = 0
    for act in _acts(n, 50, seed=1):
        oa, ra, da, _ = stock.step(act)
        ob, rb, db, _ = lat.step(act)
        assert _same(oa, ob) and _same(ra, rb) and torch.equal(da, db)
        dones += int(da.sum())
    assert dones > 0                                   # auto-resets happened
    assert torch.equal(stock.debug_records(), lat.debug_records())


def _run_schedule(n, steps, delays_at, reset_at=None, seed=2):
    """Raw joint targets within 0.1 rad of standing (joint_act), auto_reset off: each step of a latency context against a stock
    context driven by tick(targets, 1) with the per-tick targets of the numpy schedule.  delays_at(t) -> [n] delays of step t
    (None: unchanged; the stock path until the first delays); reset_at: {t: mask} explicit resets before step t, mirrored in the
    reference."""
    lat, ref = _mk(n, joint_act=True, auto_reset=False), _mk(n, joint_act=True, auto_reset=False)
    lat.reset(); ref.reset()
    S = int(lat.cfg.substeps)
    sched, last = None, np.zeros((n, 18), np.float32)     # a fresh context's last targets are the reset-pose hold target 0
    differs = 0
    for t, act in enumerate(_acts(n, steps, seed=seed, amp=0.1)):
        if reset_at and t in reset_at:
            lat.reset(reset_at[t]); ref.reset(reset_at[t])
        d = delays_at(t)
        if d is not None:
            if sched is None:                # the first call seeds the history with the robots' last targets
                sched = CommandSchedule(n, S, last)
            lat.set_env_latency(d)
            dn = d.cpu().numpy()
        ept = lat.get_state()[2][:, 12].cpu().numpy().astype(np.int64)
        raw = act.cpu().numpy()
        targets = sched.step(raw, dn, ept) if sched is not None else np.repeat(raw[None], S, 0)
        differs += int((targets != raw[None]).any(axis=(0, 2)).sum())
        last = raw
        lat.step(act)
        for k in range(S):
            ref.tick(torch.from_numpy(targets[k]).cuda(), 1)
        for a, b in zip(_physics(lat), _physics(ref)):
            assert torch.equal(a, b), t
    assert differs > n                      # the delays did act
    assert torch.equal(lat.get_env_latency().cpu(), torch.as_tensor(dn))
    return lat


def test_delayed_steps_follow_the_schedule():
    """2,048 robots with delays cycling through 0..8 ticks, 30 steps: bit-identical to the stock ticks with scheduled targets."""
    n = 2048
    d = torch.arange(n, device="cuda", dtype=torch.int32) % 9
    _run_schedule(n, 30, lambda t: d if t == 0 else None)


def test_switched_on_mid_episode_keeps_the_last_command():
    """Ten stock steps, then delays 0..8 set mid-episode: the first delayed ticks apply each robot's last command (the history
    is seeded from its last servo targets), not the hold target 0, and every step stays bit-identical to the schedule."""
    n = 2048
    d = torch.arange(n, device="cuda", dtype=torch.int32) % 9
    lat = _run_schedule(n, 25, lambda t: d if t == 10 else None, seed=14)
    t, h, has = lat._get_env_latency()
    assert has and torch.equal(t, d)


def test_reset_forgets_the_history():
    """As above with an explicit reset of a third of the robots at step 12: their delayed ticks apply the hold target 0 until the
    history has refilled."""
    n = 2048
    d = torch.arange(n, device="cuda", dtype=torch.int32) % 9
    mask = torch.arange(n, device="cuda") % 3 == 1
    _run_schedule(n, 30, lambda t: d if t == 0 else None, reset_at={12: mask})


def test_auto_reset_starts_from_a_fresh_history():
    """Agent-space actions with auto-reset: every robot whose first episode ended at the most common step t0 is, at the end,
    in exactly the state of a fresh context that was reset and fed the actions after t0 with the same delays."""
    n, steps = 2048, 30
    d = _delays(n, seed=4)
    a, b = _mk(n), _mk(n)
    a.set_env_latency(d); b.set_env_latency(d)
    a.reset(); b.reset()
    acts = _acts(n, steps, seed=5)
    first = torch.full((n,), -1, dtype=torch.int64, device="cuda")
    for t, act in enumerate(acts):
        _, _, done, _ = a.step(act)
        first = torch.where((first < 0) & done, torch.full_like(first, t), first)
    ok = first[(first >= 0) & (first < steps - 5)]
    assert ok.numel() > 0
    t0 = int(torch.mode(ok).values)
    sel = first == t0
    assert int(sel.sum()) >= 8
    for act in acts[t0 + 1:]:
        b.step(act)
    for x, y in zip(a.get_state(), b.get_state()):
        assert torch.equal(x[sel], y[sel])


def test_delays_may_change_every_step():
    """New random delays before every step still follow the schedule."""
    n = 2048
    _run_schedule(n, 30, lambda t: _delays(n, seed=100 + t), seed=6)


def test_batch_position_and_step_path_do_not_matter():
    """Permuting the robots together with their delays and actions permutes every output bit for bit; step_host (private
    streams, pipelined ranges) equals step."""
    n, steps = 8192, 20
    d = _delays(n, seed=7)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(0)).cuda()
    a, p, h = _mk(n), _mk(n), _mk(n)
    a.set_env_latency(d); p.set_env_latency(d[perm]); h.set_env_latency(d)
    a.reset(); p.reset(); h.reset()
    obs_h = np.zeros((n, 26), np.float32); rew_h = np.zeros(n, np.float32); done_h = np.zeros(n, np.uint8)
    dones = 0
    for act in _acts(n, steps, seed=8):
        oa, ra, da, _ = a.step(act)
        op, rp, dp, _ = p.step(act[perm])
        assert _same(oa[perm], op) and _same(ra[perm], rp) and torch.equal(da[perm], dp)
        h.step_host(np.ascontiguousarray(act.cpu().numpy()), obs_h, rew_h, done_h)
        assert _same(oa.cpu(), torch.from_numpy(obs_h)) and _same(ra.cpu(), torch.from_numpy(rew_h))
        assert torch.equal(da.cpu(), torch.from_numpy(done_h).bool())
        dones += int(da.sum())
    assert dones > 0
    assert torch.equal(a.debug_records(), h.debug_records())


def test_snapshots_continue_bit_for_bit(tmp_path):
    """save_state mid-run, load_state into a fresh context: the next steps are identical, with the delays and history restored.
    A snapshot without a latency table restores zero delays."""
    n = 4096
    d = _delays(n, seed=9)
    a = _mk(n)
    a.set_env_latency(d)
    a.reset()
    acts = _acts(n, 20, seed=10)
    for act in acts[:10]:
        a.step(act)
    path = str(tmp_path / "snap.pt")
    a.save_state(path)
    b = _mk(n)
    b.load_state(path)
    assert torch.equal(b.get_env_latency(), d)
    ha, hb = a._get_env_latency()[1], b._get_env_latency()[1]
    assert torch.equal(ha, hb)
    for act in acts[10:]:
        oa, ra, da, _ = a.step(act)
        ob, rb, db, _ = b.step(act)
        assert _same(oa, ob) and _same(ra, rb) and torch.equal(da, db)
    assert torch.equal(a.debug_records(), b.debug_records())
    plain = _mk(n)
    plain.reset()
    plain.save_state(path)
    b.load_state(path)
    assert int(b.get_env_latency().abs().sum()) == 0


def test_accessors_validation_tick_and_launch_count():
    n = 256
    env = _mk(n)
    # no table: zero delays, the last targets (the hold target 0 after creation) as history, and no table reported
    t, h, has = env._get_env_latency()
    assert not has and int(t.abs().sum()) == 0 and int((h != 0).sum()) == 0
    assert env.max_latency_ticks == 2 * int(env.cfg.substeps) == 8
    d = _delays(n, seed=11)
    env.set_env_latency(d)
    assert torch.equal(env.get_env_latency(), d) and env.get_env_latency().dtype == torch.int32
    env.set_env_latency(np.arange(n) % 9)
    assert torch.equal(env.get_env_latency().cpu(), torch.arange(n, dtype=torch.int32) % 9)
    env.set_env_latency(3)
    assert bool((env.get_env_latency() == 3).all())
    env.set_env_latency([2.0] * n)                          # integral floats are integers
    assert bool((env.get_env_latency() == 2).all())
    hist = torch.randn((n, 2, 18), device="cuda")
    env.set_env_latency(5, hist)
    assert torch.equal(env._get_env_latency()[1], hist)
    for bad in (torch.zeros(n + 1, dtype=torch.int32), torch.zeros((n, 1), dtype=torch.int32), [1.5] * n, -1, 9,
                torch.full((n,), float("nan")), torch.ones(n, dtype=torch.bool)):
        with pytest.raises(ValueError):
            env.set_env_latency(bad)
    with pytest.raises(ValueError):
        env.set_env_latency(0, torch.zeros((n, 18)))
    assert bool((env.get_env_latency() == 5).all())           # a refused call changed nothing
    # tick() is raw physics: the same as a context without latency, and it leaves the history alone
    ref = _mk(n)
    env.reset(); ref.reset()
    tg = _acts(n, 1, seed=12, amp=0.1)[0]
    h0 = env._get_env_latency()[1].clone()
    env.tick(tg, 3); ref.tick(tg, 3)
    assert torch.equal(env.debug_records(), ref.debug_records())
    assert torch.equal(env._get_env_latency()[1], h0)
    # a step still launches 13 kernels (k_dyn, k_rank, k_solve per tick, then k_post)
    l0, r0 = env.launches, ref.launches
    act = _acts(n, 1, seed=13)[0]
    env.step(act); ref.step(act)
    assert env.launches - l0 == ref.launches - r0 == 13
