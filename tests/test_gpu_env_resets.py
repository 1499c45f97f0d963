"""Per-robot reset states (plen_settle_env_resets / plen_set_env_resets, PlenVecEnv.settle_resets) on the GPU: nominal rows are
the shared snapshot bit for bit, a row is the reference's reset procedure run under the robot's own parameters (against plen_tick
and against the float64 oracle), every reset path restores the robot's own row at every launch geometry, the settle leaves the
running state alone, rows depend neither on batch position nor on batch size, snapshots carry the rows, and bad arguments are
refused."""
import numpy as np
import pytest

from resets_util import oracle_settle, start_qpos

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

PLEN_E_STATE = -3


def _mk(n, **kw):
    from plen_ml_walk_b200.urdf_loader import packaged_model
    from plen_ml_walk_b200.vec_env import PlenVecEnv
    kw.setdefault("model", packaged_model())
    return PlenVecEnv(n, device="cuda:0", **kw)


def _bits(t):
    return t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t


def _eq(a, b):
    """bit for bit (NaN payloads and the sign of zero included)"""
    return a.shape == b.shape and bool(torch.equal(_bits(a), _bits(b)))


def _acts(n, steps, seed, amp=1.0):
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    return [torch.empty((n, 18), device="cuda").uniform_(-amp, amp, generator=g) for _ in range(steps)]


def _params(n, seed):
    """random friction / force / gain scales, body mass scales, torso payloads and command delays for n robots"""
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    u = lambda shape, lo, hi: torch.empty(shape, device="cuda").uniform_(lo, hi, generator=g)
    pay = u((n, 4), -0.02, 0.02)
    pay[:, 0] = u((n,), 0.0, 0.1)
    return dict(fric=u((n,), 0.6, 1.4), force=u((n,), 0.7, 1.3), gain=u((n,), 0.7, 1.3), mass=u((n, 19), 0.8, 1.25), pay=pay,
                lat=torch.randint(0, 9, (n,), device="cuda", generator=g))


def _apply(env, p, idx=None):
    s = (lambda t: t) if idx is None else (lambda t: t[idx].contiguous())
    env.set_env_scales(friction=s(p["fric"]), motor_force=s(p["force"]), motor_gain=s(p["gain"]))
    env.set_env_mass(s(p["mass"]), s(p["pay"]))
    env.set_env_latency(s(p["lat"]))


def _poses(n, seed):
    rng = np.random.default_rng(seed)
    return np.stack([rng.uniform(-1, 1, n), rng.uniform(-1, 1, n), rng.uniform(0.152, 0.17, n),
                     rng.uniform(-np.pi, np.pi, n)], 1).astype(np.float32)


def _distinct_yaw(n):
    p = np.zeros((n, 4), np.float32)
    p[:, 2] = 0.158
    p[:, 3] = np.linspace(-3.0, 3.0, n) if n > 1 else -1.0
    return p


@pytest.mark.parametrize("manifold", [0, 1])
def test_nominal_rows_are_the_shared_snapshot(manifold):
    """4,096 robots: settle_resets() without parameters gives every robot exactly the shared snapshot (what a fresh context's
    get_env_resets reports, return value 0), and 50 random-action steps with auto-resets then equal a stock context bit for bit.
    After clear_env_resets the same holds for a context whose rows were not nominal."""
    n = 4096
    ov = {"sole_manifold": manifold}
    stock, settled, cleared = _mk(n, config_overrides=ov), _mk(n, config_overrides=ov), _mk(n, config_overrides=ov)
    ref, has = stock._get_env_resets()
    assert not has
    settled.settle_resets()
    got, has = settled._get_env_resets()
    assert has
    for a, b in zip(ref, got):
        assert (a is None and b is None) or _eq(a, b)
    # non-nominal rows, then cleared
    cleared.set_env_scales(friction=torch.full((n,), 0.6, device="cuda"))
    cleared.settle_resets(start_pose=_distinct_yaw(n))
    cleared.set_env_scales(friction=torch.ones(n, device="cuda"))
    assert not _eq(cleared.get_env_resets()[3], ref[3])
    cleared.clear_env_resets()
    assert not cleared._get_env_resets()[1]
    envs = (stock, settled, cleared)
    for e in envs:
        e.reset()
    dones = 0
    for act in _acts(n, 50, seed=1):
        outs = [e.step(act) for e in envs]
        o0, r0, d0, i0 = outs[0]
        for o, r, d, i in outs[1:]:
            assert _eq(o, o0) and _eq(r, r0) and torch.equal(d, d0)
            assert _eq(i["terminal_obs"], i0["terminal_obs"]) and torch.equal(i["timeout"], i0["timeout"])
        dones += int(d0.sum())
    assert dones > 0
    for e in envs[1:]:
        assert _eq(e.debug_records(), stock.debug_records())
        if manifold:
            assert _eq(e.get_manifold(), stock.get_manifold())


@pytest.mark.parametrize("manifold", [0, 1])
def test_row_is_the_reset_procedure_under_the_robots_own_parameters(manifold):
    """2,048 robots with random scales, masses, payloads and delays (which the settle must ignore), settled from random poses:
    each row is bit for bit what a second context with the same parameters reaches by set_state(start pose) and tick(zeros,
    reset_ticks), manifolds included; and the parameters did act (rows differ from a nominal context's settled rows)."""
    n = 2048
    ov = {"sole_manifold": manifold}
    p, poses = _params(n, seed=5), _poses(n, seed=6)
    a, b, nom = _mk(n, auto_reset=False, config_overrides=ov), _mk(n, auto_reset=False, config_overrides=ov), _mk(n, config_overrides=ov)
    _apply(a, p); _apply(b, p)
    a.settle_resets(start_pose=poses)
    nom.settle_resets(start_pose=poses)
    b.set_state(start_qpos(poses), torch.zeros(n, 24), torch.zeros(n, 29))
    if manifold:
        b.set_manifold(torch.zeros(n, 52))
    b.tick(torch.zeros(n, 18), int(b.cfg.reset_ticks))
    qpos, qvel, aux, obs, man = a.get_env_resets()
    bq, bv, ba = b.get_state()
    assert _eq(qpos, bq) and _eq(qvel, bv) and _eq(aux, ba)
    if manifold:
        assert _eq(man, b.get_manifold())
    nq, nv, _, _, _ = nom.get_env_resets()
    differs = ((qvel != nv).any(1) | (qpos != nq).any(1)).float().mean().item()
    assert differs > 0.99, differs
    # the settle did not move the running states: still the snapshot
    st = a.get_state()
    fresh = _mk(1, config_overrides=ov).get_state()
    assert _eq(st[0], fresh[0].expand(n, 25)) and _eq(st[1], fresh[1].expand(n, 24))


def test_rows_against_the_float64_oracle(oracle_lib):
    """Groups of robots (nominal; friction x 0.6; force x 1.3 with gain x 0.8; every body x 1.2; a 0.05 kg payload on a base axis),
    each settled from four start poses (the default one, turned and shifted ones), against PlenOracle on the equivalent tree /
    constants settled from the same poses: observation within 1e-5 for the nominal group (the reset bound of
    test_gpu_parity.py) and 1.6e-6 for the others, 3 x the worst measured on a B200 (5.4e-7, friction x 0.6; nominal 1.9e-7,
    servo 2.2e-7, bodies 2.8e-7, payload 1.6e-7)."""
    from oracle.urdf_tree import load_tree
    from mass_util import equivalent_tree, payload_on_base_axis
    from plen_ml_walk_b200.urdf_loader import packaged_model
    tree, links = load_tree(), packaged_model().body_links
    poses = np.array([[0.0, 0.0, 0.158, 0.0], [0.2, -0.1, 0.158, 0.3], [-0.7, 0.5, 0.160, -2.0], [0.0, 0.3, 0.162, 1.0]],
                     np.float32)

    def fric(c):
        for k in ("mu_lateral", "mu_spinning", "mu_rolling"):
            setattr(c, k, getattr(c, k) * 0.6)

    def servo(c):
        c.motor_max_force *= 1.3
        c.motor_kp *= 0.8

    one, zero = np.ones(19), np.zeros(4)
    # name, (friction, force, gain), mass scale, payload, oracle setup, bound
    groups = [("nominal", (1, 1, 1), one, zero, None, 1e-5),
              ("friction x0.6", (0.6, 1, 1), one, zero, fric, 1.6e-6),
              ("force x1.3 gain x0.8", (1, 1.3, 0.8), one, zero, servo, 1.6e-6),
              ("bodies x1.2", (1, 1, 1), np.full(19, 1.2), zero, None, 1.6e-6),
              ("payload 0.05 kg", (1, 1, 1), one, payload_on_base_axis(tree, 0.05, 0, 0.01), None, 1.6e-6)]
    per = poses.shape[0]
    n = per * len(groups)
    sc, ms, pl = np.ones((n, 3)), np.ones((n, 19)), np.zeros((n, 4))
    for g, (_, s, m, pay, _, _) in enumerate(groups):
        sc[g * per:(g + 1) * per] = s; ms[g * per:(g + 1) * per] = m; pl[g * per:(g + 1) * per] = pay
    env = _mk(n)
    f32 = lambda x: torch.tensor(x, dtype=torch.float32, device="cuda")
    env.set_env_scales(f32(sc[:, 0]), f32(sc[:, 1]), f32(sc[:, 2]))
    env.set_env_mass(f32(ms), f32(pl))
    env.settle_resets(start_pose=np.tile(poses, (len(groups), 1)))
    obs = env.get_env_resets()[3].cpu().numpy().astype(np.float64)
    for g, (name, _, m, pay, setup, bound) in enumerate(groups):
        t = equivalent_tree(tree, links, m, pay) if (m != 1).any() or pay[0] != 0 else None
        _, ref = oracle_settle(oracle_lib, poses, tree=t, setup=setup)
        err = np.abs(obs[g * per:(g + 1) * per] - ref).max()
        print("settled row vs oracle, %s: %.2e" % (name, err))
        assert err < bound, (name, err)


@pytest.mark.parametrize("manifold", [0, 1])
def test_every_reset_path_restores_the_robots_own_row(manifold):
    """A distinct heading per robot, so that every row is recognisable: masked reset(), auto-reset after falls and the numeric
    guard (NaN base positions injected with set_state) each leave the robot in its own row -- record, observation, manifolds -- and a
    faulted robot's terminal observation is its row's observation."""
    n = 1024
    env = _mk(n, config_overrides={"sole_manifold": manifold})
    env.settle_resets(start_pose=_distinct_yaw(n))
    rq, rv, ra, ro, rm = env.get_env_resets()

    def check(idx):
        q, v, a = env.get_state()
        assert _eq(q[idx], rq[idx]) and _eq(v[idx], rv[idx]) and _eq(a[idx], ra[idx])
        if manifold:
            assert _eq(env.get_manifold()[idx], rm[idx])

    env.reset()
    check(slice(None))
    assert _eq(env._obs, ro)
    acts = _acts(n, 40, seed=7)
    for act in acts[:5]:
        env.step(act)
    mask = torch.zeros(n, dtype=torch.bool, device="cuda"); mask[::3] = True
    obs = env.reset(mask)
    check(mask)
    assert _eq(obs[mask], ro[mask])
    # auto-reset after falls
    seen = 0
    for act in acts[5:]:
        obs, _, done, info = env.step(act)
        if bool(done.any()):
            check(done)
            assert _eq(obs[done], ro[done])
            seen += int(done.sum())
    assert seen > n // 4
    # numeric guard: a NaN base position survives the step (a NaN velocity need not: the velocity clamp's fmin / fmax can
    # replace it by a finite value within the ticks)
    before = env.fault_count()
    q, v, a = env.get_state()
    bad = torch.zeros(n, dtype=torch.bool, device="cuda"); bad[1::5] = True
    q = q.clone(); q[bad, 0] = float("nan")
    env.set_state(q, v, a)
    obs, rew, done, info = env.step(acts[0])
    assert bool(done[bad].all()) and env.fault_count() - before == int(bad.sum())
    check(bad)
    assert _eq(obs[bad], ro[bad]) and _eq(info["terminal_obs"][bad], ro[bad])
    assert bool((rew[bad] == -100).all())


@pytest.mark.parametrize("n", [1, 37, 2085, 9000, 40000])
def test_launch_geometry(n):
    """Every robot that is reset in a step gets its own row's observation, through plen_step (two ranges from 2,048 robots on)
    and plen_step_host (up to four ranges): a range that read its rows from the batch's start would fail.  max_episode_steps 4
    makes every robot reset at least every fourth step."""
    ov = {"max_episode_steps": 4}
    dev, host = _mk(n, config_overrides=ov), _mk(n, config_overrides=ov)
    for e in (dev, host):
        e.settle_resets(start_pose=_distinct_yaw(n))
        e.reset()
    ro = dev.get_env_resets()[3]
    assert _eq(host.get_env_resets()[3], ro)
    obs_h = torch.empty((n, 26), pin_memory=True); rew_h = torch.empty(n, pin_memory=True)
    done_h = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    reset_dev = reset_host = 0
    for act in _acts(n, 9, seed=8, amp=0.5):
        obs, _, done, _ = dev.step(act)
        assert _eq(obs[done], ro[done])
        reset_dev += int(done.sum())
        host.step_host(act.cpu().contiguous(), obs_h, rew_h, done_h)
        dh = done_h.bool()
        assert _eq(obs_h[dh], ro.cpu()[dh])
        reset_host += int(dh.sum())
    assert reset_dev >= 2 * n and reset_host >= 2 * n


def test_settle_leaves_the_running_state_alone():
    """Records, manifolds, the command history and the delays are bit-identical across a mid-run settle_resets(); and with nominal
    parameters a run with that call equals one without, step for step."""
    n = 4096
    ov = {"sole_manifold": 1}
    a, b = _mk(n, config_overrides=ov), _mk(n, config_overrides=ov)
    d = torch.randint(0, 9, (n,), device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    for e in (a, b):
        e.set_env_latency(d)
        e.reset()
    acts = _acts(n, 40, seed=10)
    for act in acts[:10]:
        a.step(act); b.step(act)
    rec, man, (lt, lh, _) = a.debug_records(), a.get_manifold(), a._get_env_latency()
    l0 = a.launches
    a.settle_resets()
    assert a.launches - l0 == 3 * int(a.cfg.reset_ticks) + 2     # reset_ticks ticks of (k_dyn, k_rank, k_solve), start, pack
    lt2, lh2, _ = a._get_env_latency()
    assert _eq(a.debug_records(), rec) and _eq(a.get_manifold(), man) and _eq(lt2, lt) and _eq(lh2, lh)
    assert _eq(a.get_env_latency(), d.to(torch.int32))
    dones = 0
    for act in acts[10:]:
        l0 = a.launches
        oa, ra, da, ia = a.step(act)
        ob, rb, db, ib = b.step(act)
        assert a.launches - l0 == 26          # still 13 per range, two ranges
        assert _eq(oa, ob) and _eq(ra, rb) and torch.equal(da, db) and _eq(ia["terminal_obs"], ib["terminal_obs"])
        dones += int(da.sum())
    assert dones > 0
    assert _eq(a.debug_records(), b.debug_records()) and _eq(a.get_manifold(), b.get_manifold())


def test_rows_do_not_depend_on_batch_position_or_size():
    """Permuting the robots' parameters and poses permutes the rows bit for bit, and a 1-robot context's row equals the same
    robot's row in a 4,096-robot context."""
    n = 4096
    p, poses = _params(n, seed=11), _poses(n, seed=12)
    perm = torch.randperm(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(13))
    a, b = _mk(n), _mk(n)
    _apply(a, p); _apply(b, p, perm)
    a.settle_resets(start_pose=poses)
    b.settle_resets(start_pose=poses[perm.cpu().numpy()])
    ra, rb = a.get_env_resets(), b.get_env_resets()
    for x, y in zip(ra[:4], rb[:4]):
        assert _eq(x[perm], y)
    for k in (0, 1777, n - 1):
        one = _mk(1)
        _apply(one, p, torch.tensor([k], device="cuda"))
        one.settle_resets(start_pose=poses[k:k + 1])
        for x, y in zip(ra[:4], one.get_env_resets()[:4]):
            assert _eq(x[k:k + 1], y)


def test_snapshots_carry_the_rows(tmp_path):
    """save_state, then 100 steps with auto-resets, equals load_state into a fresh context with the same parameters followed by
    the same steps, bit for bit; loading a snapshot without rows clears the table."""
    n = 2048
    ov = {"sole_manifold": 1}
    p, poses = _params(n, seed=14), _poses(n, seed=15)
    a = _mk(n, config_overrides=ov)
    _apply(a, p)
    a.settle_resets(start_pose=poses)
    a.reset()
    acts = _acts(n, 110, seed=16)
    for act in acts[:10]:
        a.step(act)
    path = str(tmp_path / "snap.pt")
    a.save_state(path)
    b = _mk(n, config_overrides=ov)
    _apply(b, p)
    b.load_state(path)
    for x, y in zip(a.get_env_resets(), b.get_env_resets()):
        assert _eq(x, y)
    dones = 0
    for act in acts[10:]:
        oa, ra, da, ia = a.step(act)
        ob, rb, db, ib = b.step(act)
        assert _eq(oa, ob) and _eq(ra, rb) and torch.equal(da, db)
        assert _eq(ia["terminal_obs"][da], ib["terminal_obs"][db])
        dones += int(da.sum())
    assert dones > n // 2
    for x, y in zip(a.get_state(), b.get_state()):
        assert _eq(x, y)
    plain = str(tmp_path / "plain.pt")
    _mk(n, config_overrides=ov).save_state(plain)
    b.load_state(plain)
    assert not b._get_env_resets()[1]


def test_argument_checks():
    """ValueError on start poses of a wrong shape or with non-finite values; PLEN_E_STATE for manifolds without sole_manifold."""
    import ctypes as C
    n = 8
    env = _mk(n)
    for bad in (np.zeros(3), np.zeros((n, 3)), np.zeros((n - 1, 4)), np.zeros((n, 4, 1))):
        with pytest.raises(ValueError):
            env.settle_resets(start_pose=bad)
    for v in (np.nan, np.inf, -np.inf):
        pose = np.tile([0.0, 0.0, 0.158, 0.0], (n, 1)); pose[3, 3] = v
        with pytest.raises(ValueError):
            env.settle_resets(start_pose=pose)
    with pytest.raises(ValueError):
        env.set_env_resets(qpos=np.zeros((n, 24)))
    assert not env._get_env_resets()[1]           # nothing was allocated by the refused calls
    man = torch.zeros((n, 52), device="cuda")
    st = env._stream()
    assert env.lib.plen_set_env_resets(env._ctx, None, None, None, C.c_void_p(man.data_ptr()), st) == PLEN_E_STATE
    assert env.lib.plen_get_env_resets(env._ctx, None, None, None, None, C.c_void_p(man.data_ptr()), st) == PLEN_E_STATE
    with pytest.raises(RuntimeError):
        env.set_env_resets(man=man)
    assert env.get_env_resets()[4] is None
    env.clear_env_resets()                        # no table: a no-op
