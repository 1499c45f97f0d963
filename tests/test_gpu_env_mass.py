"""Per-robot mass randomisation (plen_set_env_mass / PlenVecEnv.set_env_mass, SURVEY.md 8f-3) on the GPU: unit rows are the
stock robot bit for bit, doubled masses are exactly the stock dynamics in other units, scaled robots match contexts built
from an equivalent model and the float64 oracle on an equivalent tree, the ground carries the robot's weight, and the
result depends neither on batch position nor on the step path."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

G, DT = 9.81, 1.0 / 240.0


def _mk(n, **kw):
    from plen_ml_walk_b200.urdf_loader import packaged_model
    from plen_ml_walk_b200.vec_env import PlenVecEnv
    kw.setdefault("model", packaged_model())
    return PlenVecEnv(n, device="cuda:0", **kw)


def _same(a, b):
    return bool(torch.equal(a, b) or torch.equal(torch.nan_to_num(a.float(), nan=1234.5), torch.nan_to_num(b.float(), nan=1234.5)))


def _rand_mass(n, seed, payload_mass=0.08):
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    s = torch.empty((n, 19), device="cuda").uniform_(0.7, 1.4, generator=g)
    p = torch.empty((n, 4), device="cuda").uniform_(-0.03, 0.03, generator=g)
    p[:, 0] = torch.empty(n, device="cuda").uniform_(0.0, payload_mass, generator=g)
    return s, p


def _acts(n, steps, seed, amp=1.0):
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    return [torch.empty((n, 18), device="cuda").uniform_(-amp, amp, generator=g) for _ in range(steps)]


def test_unit_mass_rows_are_bit_identical_to_the_stock_path():
    """Scale 1, payload 0: 4,096 robots, 50 random-action steps with auto-reset, obs / reward / done / state records equal to a
    context that never called the setter (which runs the stock k_dyn instance)."""
    n = 4096
    stock, unit = _mk(n), _mk(n)
    unit.set_env_mass(torch.ones(n, 19), torch.zeros(n, 4))
    stock.reset(); unit.reset()
    dones = 0
    for act in _acts(n, 50, seed=1):
        oa, ra, da, _ = stock.step(act)
        ob, rb, db, _ = unit.step(act)
        assert _same(oa, ob) and _same(ra, rb) and torch.equal(da, db)
        dones += int(da.sum())
    assert dones > 0                                   # auto-resets happened
    assert torch.equal(stock.debug_records(), unit.debug_records())


def test_doubled_masses_are_the_stock_dynamics_in_other_units():
    """Every body x 2 and the servo force limit x 2 (set_env_scales), with the cached normal impulses doubled: every term of the
    step is homogeneous in mass and x 2 is exact in floating point, so obs and reward equal the stock robot's bit for bit through
    contact, the cached impulses stay exactly doubled and M^-1 is exactly half.  auto_reset off: a reset would restore the nominal
    impulses; robots that finish leave the comparison, so the actions are raw joint targets (joint_act) within 0.1 rad of the
    standing pose, which keep most of them on their feet (agent-space actions topple nearly all within 30 steps)."""
    n = 2048
    stock, dbl = _mk(n, auto_reset=False, joint_act=True), _mk(n, auto_reset=False, joint_act=True)
    dbl.set_env_mass(torch.full((n,), 2.0))
    dbl.set_env_scales(motor_force=torch.full((n,), 2.0, device="cuda"))
    stock.reset(); dbl.reset()
    for act in _acts(n, 3, seed=2, amp=0.1):
        stock.step(act)
    qpos, qvel, aux = (t.clone() for t in stock.get_state())
    aux2 = aux.clone(); aux2[:, :8] *= 2
    dbl.set_state(qpos, qvel, aux2)
    alive = torch.ones(n, dtype=torch.bool, device="cuda")
    for act in _acts(n, 25, seed=3, amp=0.1):
        oa, ra, da, _ = stock.step(act)
        ob, rb, db, _ = dbl.step(act)
        assert _same(oa[alive], ob[alive]) and _same(ra[alive], rb[alive]) and torch.equal(da[alive], db[alive])
        alive &= ~da
    assert int(alive.sum()) > n // 2
    a1, a2 = stock.get_state()[2], dbl.get_state()[2]
    assert torch.equal(2 * a1[alive, :8], a2[alive, :8]) and bool((a1[alive, :8] > 0).any())
    m1, m2 = stock.debug_dynamics()[0], dbl.debug_dynamics()[0]
    assert torch.equal(0.5 * m1[alive], m2[alive])


def _groups():
    """Four parameter groups; payloads at arbitrary offsets in the torso frame."""
    rng = np.random.default_rng(5)
    return [(np.full(19, 1.25), np.zeros(4)),
            (rng.uniform(0.6, 1.5, 19), np.array([0.03, 0.01, -0.02, 0.03])),
            (np.ones(19), np.array([0.2, -0.03, 0.02, 0.05])),
            (rng.uniform(0.8, 1.2, 19), np.array([0.08, 0.0, 0.0, -0.01]))]


def test_mass_rows_match_contexts_built_from_an_equivalent_model():
    """One free-flight env step from the same forced state against a context whose lane tables hold the scaled bodies and the
    payload folded into the torso: positions within 1e-5, M^-1 (relative to sqrt(M^-1_ii M^-1_jj)) and velocities within 1e-4
    relative.  The two contexts form the same inertias in different float32 operations (the scaling in the kernel, the folding
    in float64 before the table is rounded), and M's condition number (2e5 .. 3e5) turns those 1e-7 differences into up to
    2.2e-5 in M^-1 and 3.1e-5 in the velocities (measured on a B200); the float64 emulation holds the two to 1e-6
    (test_emu_mass.py)."""
    from mass_util import equivalent_model
    from parity_util import random_flight_state
    from plen_ml_walk_b200.urdf_loader import packaged_model
    per, groups = 16, _groups()
    n = per * len(groups)
    rng = np.random.default_rng(6)
    qpos, qvel = random_flight_state(rng, n)
    qpos, qvel = torch.tensor(qpos, dtype=torch.float32), torch.tensor(qvel, dtype=torch.float32)
    env = _mk(n, auto_reset=False)
    env.set_env_mass(torch.tensor(np.repeat([s for s, _ in groups], per, 0), dtype=torch.float32),
                     torch.tensor(np.repeat([p for _, p in groups], per, 0), dtype=torch.float32))
    env.set_state(qpos, qvel)
    act = torch.empty((n, 18), device="cuda").uniform_(-1, 1, generator=torch.Generator(device="cuda").manual_seed(7))
    minv = env.debug_dynamics()[0].cpu().numpy()
    env.step(act)
    got_q, got_v = (t.cpu().numpy() for t in env.get_state()[:2])
    worst_m, worst_q, worst_v = 0.0, 0.0, 0.0
    for g, (s, p) in enumerate(groups):
        sl = slice(g * per, (g + 1) * per)
        eq = _mk(per, auto_reset=False, model=equivalent_model(packaged_model(), s, p))
        eq.set_state(qpos[sl], qvel[sl])
        m_ref = eq.debug_dynamics()[0].cpu().numpy()
        eq.step(act[sl])
        ref_q, ref_v = (t.cpu().numpy() for t in eq.get_state()[:2])
        d = np.sqrt(np.einsum("eii,ejj->eij", m_ref, m_ref))
        worst_m = max(worst_m, float(np.abs((minv[sl] - m_ref) / d).max()))
        worst_q = max(worst_q, float(np.abs(got_q[sl] - ref_q).max()))
        worst_v = max(worst_v, float((np.abs(got_v[sl] - ref_v) / np.maximum(1.0, np.abs(ref_v))).max()))
    print("equivalent model: M^-1 rel %.2e, qpos %.2e, qvel rel %.2e" % (worst_m, worst_q, worst_v))
    assert worst_m < 1e-4 and worst_q < 1e-5 and worst_v < 1e-4


def test_mass_rows_against_oracles_on_equivalent_trees(oracle_lib):
    """Teacher-forced through contact like test_per_env_scales_against_oracles_with_scaled_constants, with its thresholds: the
    first half of the batch carries four mass groups (payloads on the base link's principal axes, where the oracle's folded base
    inertia stays diagonal), each checked against an oracle on the equivalent tree; the second half is stock."""
    from oracle.urdf_tree import load_tree
    from mass_util import equivalent_tree, payload_on_base_axis
    from parity_util import abi_from_oracle
    from plen_ml_walk_b200.urdf_loader import packaged_model
    tree, links = load_tree(), packaged_model().body_links
    rng = np.random.default_rng(12)
    groups = [(np.full(19, 0.8), payload_on_base_axis(tree, 0.05, 2, 0.01)),
              (rng.uniform(0.7, 1.4, 19), np.zeros(4)),
              (np.full(19, 1.2), payload_on_base_axis(tree, 0.1, 0, -0.01)),
              (rng.uniform(0.9, 1.1, 19), payload_on_base_axis(tree, 0.03, 1, 0.02))]
    n, h, steps, per = 64, 32, 25, 8
    oracles = [oracle_lib.PlenOracle(per, n_threads=2, tree=equivalent_tree(tree, links, s, p)) for s, p in groups]
    stock_o = oracle_lib.PlenOracle(h, n_threads=4)
    scale = np.ones((n, 19)); pay = np.zeros((n, 4))
    for g, (s, p) in enumerate(groups):
        scale[g * per:(g + 1) * per] = s; pay[g * per:(g + 1) * per] = p
    env = _mk(n, auto_reset=False)
    env.set_env_mass(torch.tensor(scale, dtype=torch.float32), torch.tensor(pay, dtype=torch.float32))
    every = oracles + [stock_o]
    for o in every:
        o.reset()
    env.reset()
    errs = []
    for t in range(steps):
        st = [o.get_state() for o in every]
        env.set_state(*abi_from_oracle({k: np.concatenate([s[k] for s in st]) for k in st[0]}))
        act = rng.uniform(-1, 1, (n, 18)).astype(np.float32)
        outs, lo = [], 0
        for o in every:
            x, _, d, _ = o.step(act[lo:lo + o.n].astype(np.float64))
            outs.append(x)
            for e in np.where(d)[0]:
                o.reset_one(int(e))
            lo += o.n
        go, _, _, _ = env.step(torch.from_numpy(act).cuda())
        errs.append(np.abs(go.cpu().numpy()[:, :24] - np.concatenate(outs)[:, :24]).max(1))
    errs = np.stack(errs)
    print("mass rows vs oracles: median err randomised %.2e stock %.2e, share < 1e-3 %.2f"
          % (np.median(errs[:, :h]), np.median(errs[:, h:]), np.mean(errs < 1e-3)))
    assert np.median(errs[:, :h]) < 1e-4 and np.median(errs[:, h:]) < 1e-4
    assert np.mean(errs < 1e-3) > 0.6


def test_the_ground_carries_the_robot_weight():
    """Standing under zero raw targets (joint_act), the normal impulses of a tick add up to the weight: the mean over ticks
    60..240 of sum(lambda_n) / (g dt) is the supported mass.  For each group its ratio to the stock robot's figure is the
    mass ratio sum(s_b m_b) + m_p over the stock mass, within a tolerance set from how closely the stock robot's own figure
    matches its mass."""
    from mass_util import BODY_LANES
    from plen_ml_walk_b200.urdf_loader import packaged_model
    model = packaged_model()
    m_body = np.array([model.mass[l] for l in BODY_LANES])
    com0 = np.array(model.com[0])
    groups = [(np.ones(19), np.zeros(4)), (np.full(19, 0.8), np.zeros(4)), (np.full(19, 1.2), np.zeros(4)),
              (np.ones(19), np.r_[0.05, com0]), (np.ones(19), np.r_[0.025, com0]),
              (np.random.default_rng(8).uniform(0.9, 1.1, 19), np.r_[0.03, com0])]
    per = 4
    n = per * len(groups)
    scale = np.repeat([s for s, _ in groups], per, 0); pay = np.repeat([p for _, p in groups], per, 0)
    env = _mk(n, auto_reset=False, joint_act=True)
    env.set_env_mass(torch.tensor(scale, dtype=torch.float32), torch.tensor(pay, dtype=torch.float32))
    env.reset()
    zero = torch.zeros((n, 18), device="cuda")
    lam = []
    for t in range(241):
        env.tick(zero, 1)
        if t >= 60:
            lam.append(env.get_state()[2][:, :8].sum(1).cpu().numpy())
    supported = np.mean(lam, 0) / (G * DT)                     # kg, per robot
    mass = scale @ m_body + pay[:, 0]
    stock = supported[:per].mean()
    stock_err = abs(stock / m_body.sum() - 1.0)
    ratio_err = np.abs((supported / stock) / (mass / m_body.sum()) - 1.0)
    print("weight: stock robot carries %.5f kg of %.5f kg (rel. err %.2e); ratio errors per group %s"
          % (stock, m_body.sum(), stock_err, [float("%.2e" % ratio_err[g * per:(g + 1) * per].max()) for g in range(len(groups))]))
    assert np.isfinite(supported).all() and stock_err < 0.02
    assert ratio_err.max() < max(2 * stock_err, 2e-3)


def test_result_does_not_depend_on_batch_position_or_step_path():
    """Randomised robots at permuted batch positions step bit-identically (auto-reset included), and at a size that runs several
    ranges plen_step_host returns what plen_step returns with the mass table set."""
    n = 16384
    s, p = _rand_mass(n, seed=9)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(10)).cuda()
    a, b, c = _mk(n), _mk(n), _mk(n)
    a.set_env_mass(s, p); b.set_env_mass(s[perm], p[perm]); c.set_env_mass(s, p)
    a.reset(); b.reset(); c.reset()
    h_obs = torch.empty((n, 26)).pin_memory(); h_rew = torch.empty(n).pin_memory()
    h_done = torch.empty(n, dtype=torch.uint8).pin_memory()
    for act in _acts(n, 20, seed=11):
        oa, ra, da, _ = a.step(act)
        ob, rb, db, _ = b.step(act[perm])
        assert _same(oa[perm], ob) and _same(ra[perm], rb) and torch.equal(da[perm], db)
        torch.cuda.synchronize()
        c.step_host(act.cpu().pin_memory(), h_obs, h_rew, h_done)
        assert _same(oa.cpu(), h_obs) and _same(ra.cpu(), h_rew) and torch.equal(da.cpu(), h_done.bool())
    assert torch.equal(a.debug_records()[perm], b.debug_records())


def test_python_surface_round_trip_snapshots_and_argument_checks(tmp_path):
    n = 3000
    a = _mk(n)
    s0, p0 = a.get_env_mass()
    assert bool((s0 == 1).all()) and bool((p0 == 0).all()) and s0.shape == (n, 19) and p0.shape == (n, 4)
    assert len(a.body_links) == 19 and a.body_links[0][0] == "torso"
    s, p = _rand_mass(n, seed=13)
    a.set_env_mass(s, p)
    gs, gp = a.get_env_mass()
    assert torch.equal(gs, s) and torch.equal(gp, p)
    a.set_env_mass(payload=torch.zeros(n, 4))                   # None leaves the other part as it is
    gs, gp = a.get_env_mass()
    assert torch.equal(gs, s) and bool((gp == 0).all())
    a.set_env_mass(torch.full((n,), 1.1))                       # [N]: one factor for every body
    assert bool((a.get_env_mass()[0] == torch.tensor(1.1)).all())
    a.set_env_mass(s, p)
    for act in _acts(n, 10, seed=14):
        a.step(act)
    path = str(tmp_path / "mass_state.pt")
    a.save_state(path)
    b = _mk(n)
    b.reset()
    b.load_state(path)
    assert torch.equal(b.get_env_mass()[0], s) and torch.equal(b.get_env_mass()[1], p)
    for act in _acts(n, 4, seed=15):
        ra, rb = a.step(act), b.step(act)
        assert _same(ra[0], rb[0]) and _same(ra[1], rb[1]) and torch.equal(ra[2], rb[2])
    # a snapshot without a mass entry (a context that never set one) restores unit values
    plain = _mk(n)
    plain.reset()
    p2 = str(tmp_path / "plain.pt")
    plain.save_state(p2)
    assert torch.load(p2)["mass"] is None
    b.load_state(p2)
    assert bool((b.get_env_mass()[0] == 1).all()) and bool((b.get_env_mass()[1] == 0).all())
    for bad in (dict(mass_scale=torch.ones(n, 18)), dict(mass_scale=torch.zeros(n)), dict(mass_scale=torch.full((n,), float("nan"))),
                dict(mass_scale=-torch.ones(n, 19)), dict(payload=torch.ones(n, 3)), dict(payload=-torch.ones(n, 4)),
                dict(payload=torch.full((n, 4), float("inf")))):
        with pytest.raises(ValueError):
            a.set_env_mass(**bad)
