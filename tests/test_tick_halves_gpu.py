"""GPU tests of the two halves of a physics tick, each on its own and robot by robot, against float64 references.

k_dyn writes the solve record (SR_*), the extension record of box contacts (XR_*) and a sort key per robot; k_rank groups the
robots by key; k_solve / k_solve_x run the projected Gauss-Seidel (PGS) on those records.  The harness library
(tests/cuda/tick_harness.cu, the library's own source with th_dyn / th_rank / th_solve exported) lets these tests read and
write that buffer between the halves, and the float64 build of the warp emulation (tests/emu/emu_halves.cpp) evaluates the
same device source on the same inputs.  Each half is a deterministic function of its inputs: k_dyn is smooth apart from a
few discrete decisions, and PGS capped at k sweeps without early exit (residual_threshold < 0) is a composition of
continuous clamps, so every bound here is per element or per robot, never a quantile.  The stock 50 sweeps are chaotic at
impacts; there each robot is held to its own float64 sensitivity.

Every bound is a few times the worst case measured on one B200; the measurements are quoted beside the bounds and in
DESIGN.md section 1."""
import numpy as np
import pytest
import torch

from emu_halves_util import (FAMILIES, KEY_EXT, SR_MAN, SWEEP_BOUND, EmuHalves, ext_errors, make_family, real_noise,
                             record_errors, sort_keys, structure)

pytestmark = pytest.mark.gpu

N_FAM = 192          # robots per state family
DT = 1.0 / 240.0


@pytest.fixture(scope="module")
def e64():
    return EmuHalves(double=True)


@pytest.fixture(scope="module")
def fams(oracle_lib):
    return {f: make_family(oracle_lib, f, N_FAM, seed=100 + i) for i, f in enumerate(FAMILIES)}


def _ctx(n, cfg=None):
    from tick_harness_util import TickCtx
    return TickCtx(n, cfg)


def _load(ctx, F, rec=None):
    """write a family's state records (and its scales, mass rows and manifolds) into a context"""
    ctx.state.copy_(torch.from_numpy(F["rec"] if rec is None else rec).cuda())
    if F["scales"] is not None:
        ctx.scale.copy_(torch.from_numpy(F["scales"]).cuda())
    if F["mass_scale"] is not None:
        ctx.set_mass(F["mass_scale"], F["payload"])
    if F["man"] is not None:
        ctx.man.copy_(torch.from_numpy(F["man"]).cuda())
    torch.cuda.synchronize()


def _np(t):
    return t.cpu().numpy()


def _mixed(fams, names=("contact", "fallen", "limits")):
    rec = np.concatenate([fams[f]["rec"] for f in names])
    tg = np.concatenate([fams[f]["tgt"] for f in names])
    return dict(rec=rec, tgt=tg, cfg={}, scales=None, mass_scale=None, payload=None, man=None)


# ------------------------------------------------------------------------------------------------ a. harness sanity
@pytest.mark.parametrize("merged", [1, 0])
def test_harness_halves_match_plen_tick(fams, merged):
    """th_dyn -> th_rank -> th_solve is plen_tick(..., 1) bit for bit on the same state, with the merged k_solve<true> and
    with the split k_solve<false> + k_solve_x: 5,000 robots, box contacts present."""
    F = _mixed(fams)
    n = 5000
    idx = np.arange(n) % F["rec"].shape[0]
    rec, tg = F["rec"][idx], torch.from_numpy(F["tgt"][idx]).cuda()
    a, b = _ctx(n), _ctx(n)
    try:
        a.state.copy_(torch.from_numpy(rec).cuda())
        b.state.copy_(torch.from_numpy(rec).cuda())
        a.set_solver(merge_max=n if merged else 0)
        a.tick(tg)
        b.dyn(tg)
        b.rank()
        b.solve(merged)
        torch.cuda.synchronize()
        assert int((b.key >= KEY_EXT).sum()) > 100
        assert torch.equal(a.state, b.state)
    finally:
        a.close(); b.close()


# ------------------------------------------------------------------------------------------------ b. k_dyn vs float64
# per-element bounds relative to the row's block maximum, a few times the worst case measured on a B200 over the six
# families (in brackets).  The contact right-hand sides and the servo rows subtract velocities of similar size (v* against
# the contact / target velocity), so their float32 error is larger relative to the block; v* itself is clamped at
# max_coord_velocity in the vclamp family.
REC_BOUND = dict(G=2e-4,          # 3.8e-5
                 B=5e-4,          # 1.4e-4
                 MRHS=1e-3,       # 2.1e-4
                 MD=2e-4,         # 2.1e-5
                 LDIR=0.0, Q=0.0, LAMC=0.0,
                 LRHS=2e-4,       # 3.2e-6
                 VSTAR=1.5e-3,    # 3.1e-4
                 CRHS=2.5e-3,     # 6.6e-4
                 CDINV=2e-4,      # 1.7e-5
                 CD=2e-4,         # 1.4e-5
                 PT=2e-4,         # 2.5e-7
                 BASE=2e-4)       # 2.5e-5
EXT_BOUND = 1e-4                  # Jx 4.3e-8, Bx 1.4e-5, Bb 2.0e-5, row scalars 5.5e-6
MAN_SAME = 1e-5                   # m: two sole manifolds hold the same hull vertices (vertices are millimetres apart)


def _man_diff(a, b, n):
    return np.zeros(n, bool) if a is None else np.abs(a - b).max(1) > MAN_SAME


def _structure_near_threshold(e64, F, s64, x64, k64, man64):
    """Robots whose discrete structure (key, manifold bits, box points, limit rows, contact slots, the hull vertices a sole
    manifold keeps) changes in float64 when the real-valued words of their float32 state record are moved by 2e-5
    relative (3 draws; about 1e-6 m at the contact points, the float32 error of k_dyn's kinematics): their deciding
    quantity (a sole vertex's distance against foot_break, a penetration's sign, a contact velocity against
    restitution_vel_threshold, a joint against its limit, a box's lowest point against 0, the lowest of nearly coplanar
    hull vertices) lies within that of its threshold, where float32 may decide either way."""
    base = structure(s64, x64, k64)
    near = np.zeros(len(base), bool)
    rng = np.random.default_rng(7)
    real = np.ones(96, bool)
    real[[35, 60, 61, 62, 63, 79]] = False       # manifold bits and integer counters
    for _ in range(3):
        rec = F["rec"].astype(np.float64)
        rec[:, real] *= 1.0 + 2e-5 * rng.choice([-1.0, 1.0], rec[:, real].shape)
        man = None if F["man"] is None else F["man"].astype(np.float64)
        s, x, k = e64.dyn(rec, F["tgt"], F["scales"], _mass_rows(F), man)
        near |= (structure(s, x, k) != base).any(1) | _man_diff(man, man64, len(base))
    return near


def _mass_rows(F):
    if F["mass_scale"] is None:
        return None
    from emu_mass_util import mass_rows
    return mass_rows(F["mass_scale"], F["payload"], dtype=np.float64)


@pytest.mark.parametrize("fam", FAMILIES)
def test_dyn_record_vs_f64(fams, e64, fam):
    """k_dyn's solve record and extension record against the float64 emulation of tick_dynamics on the same float32 state
    records and targets (per-robot scales and mass rows: the MASS instance; sole_manifold = 1 with the manifolds set).
    The discrete structure must be equal exactly, apart from robots whose deciding quantity sits within 2e-5 relative of its
    threshold (_structure_near_threshold; at most 5 % of a family; measured on a B200: at most 2 of 192, and no
    robot's structure differed).  Every continuous
    word, block by block, within REC_BOUND of its row's block maximum per element; the box-contact rows' Jx / Bx / Bb /
    scalars within EXT_BOUND of their part's maximum.  Both sides start from records filled with NaN: k_dyn must write
    exactly the words the emulation writes (the words it leaves alone, such as the padding of the base block, are never
    read), and only those are compared."""
    F = fams[fam]
    n = F["rec"].shape[0]
    ctx = _ctx(n, F["cfg"])
    try:
        _load(ctx, F)
        ctx.srec.fill_(float("nan"))
        ctx.srx.fill_(float("nan"))
        ctx.dyn(torch.from_numpy(F["tgt"]).cuda())
        torch.cuda.synchronize()
        sg, xg, kg = _np(ctx.srec).astype(np.float64), _np(ctx.srx).astype(np.float64), _np(ctx.key)
        man_g = None if F["man"] is None else _np(ctx.man).astype(np.float64)
        if F["mass_scale"] is not None:
            assert np.array_equal(_np(ctx.mass), _mass_rows(F).astype(np.float32))
    finally:
        ctx.close()
    e64.cfg.sole_manifold = F["cfg"].get("sole_manifold", 0)
    try:
        man64 = None if F["man"] is None else F["man"].astype(np.float64)
        s64, x64, k64 = e64.dyn(F["rec"], F["tgt"], F["scales"], _mass_rows(F), man64, fill=np.nan)
        written = ~np.isnan(s64), ~np.isnan(x64)
        s64, x64 = np.nan_to_num(s64), np.nan_to_num(x64)
        near = _structure_near_threshold(e64, F, s64, x64, k64, man64)
    finally:
        e64.cfg.sole_manifold = 0
    same_words = (~np.isnan(sg) == written[0]).all(1) & (~np.isnan(xg) == written[1]).all(1)
    sg, xg = np.nan_to_num(sg), np.nan_to_num(xg)
    assert np.array_equal(kg, sort_keys(sg, xg))
    same = (structure(sg, xg, kg) == structure(s64, x64, k64)).all(1) & ~_man_diff(man_g, man64, n) & same_words
    print("%s: %d / %d robots near a threshold, %d with a different structure (all near: %s)"
          % (fam, near.sum(), n, (~same).sum(), bool(near[~same].all())))
    assert near.sum() <= 0.05 * n
    assert (same | near).all()
    ok = same & ~near
    rerr = record_errors(sg[ok], s64[ok])
    xerr = ext_errors(xg[ok], x64[ok])
    print("%s record, worst element rel. to block max:" % fam, {k: "%.1e" % v.max() for k, v in rerr.items()},
          {k: "%.1e" % v.max() for k, v in xerr.items()})
    for k, v in rerr.items():
        assert v.max() <= REC_BOUND[k], k
    for k, v in xerr.items():
        assert v.max() < EXT_BOUND, k
    if fam == "fallen":
        assert (kg >= KEY_EXT).mean() > 0.5
    if fam == "limits":
        assert (sg[:, 1216:1248] != 0).any(1).sum() > N_FAM // 2
    if fam == "manifold":
        assert (sg[:, SR_MAN] != 0).mean() > 0.5


# ------------------------------------------------------------------------------------------------ c. k_solve vs float64
# per-robot bounds on |GPU - float64| of k capped sweeps on the GPU's own record: velocities (rad/s, m/s) and cached impulses
# (emu_halves_util.SWEEP_BOUND; measured on a B200: 7.7e-5 / 3.3e-4 / 5.2e-4 / 7.7e-4, poses 3.3e-7 / 1.4e-6 / 2.2e-6 / 3.2e-6)
POSE_WORDS = np.r_[32:35, 38:60]


@pytest.fixture(scope="module")
def solve_set(fams):
    """contact states, fallen poses (EXT robots) and limit rows in one batch, after th_dyn: (ctx, state0, srec, srx, keys)"""
    F = _mixed(fams)
    ctx = _ctx(F["rec"].shape[0])
    _load(ctx, F)
    ctx.dyn(torch.from_numpy(F["tgt"]).cuda())
    torch.cuda.synchronize()
    out = (ctx, ctx.state.clone(), _np(ctx.srec), _np(ctx.srx), _np(ctx.key))
    yield out
    ctx.close()


def _gpu_solve(ctx, state0, merged, iterations, threshold):
    ctx.state.copy_(state0)
    ctx.set_solver(iterations, threshold)
    ctx.rank()
    ctx.solve(merged)
    torch.cuda.synchronize()
    out = _np(ctx.state)
    ctx.set_solver()
    return out


@pytest.mark.parametrize("its", [1, 2, 4, 8])
def test_solve_capped_sweeps_vs_f64(solve_set, e64, its):
    """k_solve on the GPU's own records, capped at `its` sweeps without early exit, against emu_solve in float64 on the same
    records: every robot's velocities and cached impulses within SWEEP_BOUND[its], its pose within SWEEP_BOUND[its] * dt +
    2e-6, the iteration word exact -- in both solve modes, over EXT robots, limit rows and 8-point robots."""
    ctx, state0, srec, srx, keys = solve_set
    man = srec[:, SR_MAN].astype(np.int64)
    assert (keys >= KEY_EXT).sum() > 50 and ((man & 255) == 255).sum() > 0 and (srec[:, 1216:1248] != 0).any(1).sum() > 50
    ref = _np(state0).astype(np.float64)
    try:
        e64.set_solver(its, -1.0)
        e64.solve(ref, srec, srx, keys)
    finally:
        e64.set_solver(50, 1e-7)
    for merged in (1, 0):
        got = _gpu_solve(ctx, state0, merged, its, -1.0)
        dv = np.abs(got[:, :32] - ref[:, :32]).max(1)
        dq = np.abs(got[:, POSE_WORDS] - ref[:, POSE_WORDS]).max(1)
        print("%d sweeps, merged %d: worst robot velocity / impulse %.2e, pose %.2e" % (its, merged, dv.max(), dq.max()))
        assert (got[:, 79] == its).all()
        assert np.array_equal(got[:, 35], ref[:, 35])
        assert dv.max() < SWEEP_BOUND[its]
        assert dq.max() < SWEEP_BOUND[its] * DT + 2e-6


# stock 50 sweeps: |GPU - float64| <= SENS_C * (the robot's own float64 sensitivity) + SENS_FLOOR
SENS_C, SENS_FLOOR = 4.0, 2e-3


def test_solve_stock_sweeps_vs_own_sensitivity(solve_set, e64):
    """The stock 50-sweep solve with early exit, robot by robot: the GPU's error against the float64 solve of the same record
    must stay within SENS_C x that robot's float64 sensitivity (the largest change of its velocities over 3 draws of 1-ulp
    noise on the real-valued record words) plus SENS_FLOOR.  Measured on a B200: (error - floor) / sensitivity at most 1.70;
    robots with a sensitivity under 1e-5 within 1.8e-4; the chaotic ones reach errors of 47 rad/s against sensitivities of
    58."""
    ctx, state0, srec, srx, keys = solve_set
    ref = _np(state0).astype(np.float64)
    e64.solve(ref, srec, srx, keys)
    rng = np.random.default_rng(5)
    sens = np.zeros(ref.shape[0])
    for _ in range(3):
        a, b = real_noise(srec.astype(np.float64), srx.astype(np.float64), rng, 2.0 ** -24)
        r = _np(state0).astype(np.float64)
        e64.solve(r, a, b, keys)
        sens = np.maximum(sens, np.abs(r[:, :24] - ref[:, :24]).max(1))
    for merged in (1, 0):
        got = _gpu_solve(ctx, state0, merged, 50, 1e-7)
        err = np.abs(got[:, :24] - ref[:, :24]).max(1)
        ratio = (err - SENS_FLOOR) / np.maximum(sens, 1e-30)
        print("50 sweeps, merged %d: worst error %.2e, worst sensitivity %.2e, worst (err - floor) / sens %.2f, "
              "worst error of robots with sens < 1e-5: %.2e" % (merged, err.max(), sens.max(), ratio.max(),
                                                               err[sens < 1e-5].max() if (sens < 1e-5).any() else 0.0))
        assert (err <= SENS_C * sens + SENS_FLOOR).all()


# ------------------------------------------------------------------------------------------------ d. adversarial grouping
def test_solver_group_does_not_change_a_robot(solve_set):
    """A robot's result does not depend on the robots it is solved with (default threshold, where converged robots freeze):
    probes solved alone with 7 invalid slots, next to robots with 8 sole points / box contacts / limit rows that converge
    later, next to airborne robots that converge earlier, and a non-EXT probe inside an EXT group, have bit-identical state
    words 0-79 in every grouping and both solve modes.  Groups k_rank would never form; a plain group never holds an EXT
    robot."""
    ctx, state0, srec, srx, keys = solve_set
    n = keys.shape[0]
    man = srec[:, SR_MAN].astype(np.int64)
    lim = (srec[:, 1216:1248] != 0).any(1)
    ext = keys >= KEY_EXT
    heavy_x = list(np.where(ext)[0][:3]) + list(np.where((man & 255) == 255)[0][:2]) + list(np.where(lim & ~ext)[0][:2])
    light = list(np.where((man == 0) & ~lim & ~ext)[0][:7])
    heavy_plain = list(np.where(~ext & (man != 0))[0][-4:]) + list(np.where(lim & ~ext)[0][-3:])
    assert len(heavy_x) == 7 and len(light) == 7 and len(heavy_plain) == 7
    probes = [int(np.where(~ext & (man != 0))[0][0]), int(np.where(lim & ~ext)[0][0]), int(np.where(ext)[0][-1])]
    for p in probes:
        others = dict(alone=([n + j for j in range(7)], ext[p]), light=(light, ext[p]), heavy_x=(heavy_x, True))
        if not ext[p]:
            others["heavy_plain"] = (heavy_plain, False)
        for merged in (1, 0):
            res = {}
            for name, (mates, xgrp) in others.items():
                mates = [m for m in mates if m != p][:7]
                mates += [n + 7 + j for j in range(7 - len(mates))]
                group = [p] + list(mates)
                ctx.state.copy_(state0)
                ctx.perm.fill_(n)
                ctx.perm[:8] = torch.tensor(group[::-1] if name == "light" else group, dtype=torch.int32, device="cuda")
                ctx.xgroups.fill_(1 if xgrp else 0)
                ctx.solve(merged)
                torch.cuda.synchronize()
                res[name] = _np(ctx.state[p, :80]).copy()
            first = next(iter(res.values()))
            for name, r in res.items():
                assert np.array_equal(r.view(np.uint32), first.view(np.uint32)), (p, merged, name)


# ------------------------------------------------------------------------------------------------ e. k_rank exact
@pytest.mark.parametrize("n,mode", [(1, "random"), (7, "random"), (1000, "random"), (1024, "random"), (1025, "random"),
                                    (3000, "random"), (3000, "equal"), (1024, "ext")])
def test_rank_matches_stable_sort(n, mode):
    """k_rank on synthetic keys (foot-only keys, every EXT class, keys above RANK_KEY_MAX = 128): each tile's permutation is a
    numpy stable sort by class (class = 128 - min(key, 128), slots >= n last), and xgroups[t] = ceil(EXT robots of tile t / 8)."""
    rng = np.random.default_rng(n)
    if mode == "equal":
        keys = np.full(n, 57, np.uint8)
    elif mode == "ext":
        keys = rng.integers(KEY_EXT, 256, n).astype(np.uint8)
    else:
        keys = np.where(rng.random(n) < 0.1, rng.integers(KEY_EXT, 256, n), rng.integers(0, KEY_EXT, n)).astype(np.uint8)
    ctx = _ctx(n)
    try:
        ctx.key.copy_(torch.from_numpy(keys).cuda())
        ctx.perm.fill_(-1)
        ctx.xgroups.fill_(-1)
        ctx.rank()
        torch.cuda.synchronize()
        perm, xg = _np(ctx.perm), _np(ctx.xgroups)
    finally:
        ctx.close()
    for t in range((n + 1023) // 1024):
        r = np.arange(1024 * t, 1024 * (t + 1))
        cls = np.where(r < n, 128 - np.minimum(keys[np.minimum(r, n - 1)].astype(np.int64), 128), 159)
        assert np.array_equal(perm[1024 * t:1024 * (t + 1)], r[np.argsort(cls, kind="stable")])
        nx = int(((r < n) & (keys[np.minimum(r, n - 1)] >= KEY_EXT)).sum())
        assert xg[t] == (nx + 7) // 8


# ------------------------------------------------------------------------------------------------ f. whole tick vs oracle
# per robot: velocities (rad/s, m/s), pose (rad, m); measured on a B200: 9.3e-4 / 3.9e-6 at 1 sweep, 5.7e-3 / 2.4e-5 at 4
ORACLE_BOUND = {1: (4e-3, 2e-5), 4: (2e-2, 1e-4)}


@pytest.mark.parametrize("its", [1, 4])
def test_whole_tick_vs_oracle_capped_sweeps(oracle_lib, fams, its):
    """plen_tick through PlenVecEnv (no harness) one tick from oracle states against PlenOracle.tick, both capped at `its`
    sweeps without early exit: every robot within ORACLE_BOUND[its] in velocity and pose.  Contact states, fallen poses
    with box contacts and limit rows; an implementation independent of the warp emulation."""
    from emu_util import oracle_state_from_record
    from parity_util import abi_from_oracle
    from plen_ml_walk_b200.vec_env import PlenVecEnv
    F = _mixed(fams)
    n = F["rec"].shape[0]
    st = oracle_state_from_record(F["rec"])
    st["target"] = F["tgt"].astype(np.float64)
    o = oracle_lib.PlenOracle(n)
    o.cfg.solver_iterations = its
    o.cfg.residual_threshold = -1.0
    o.set_state(st)
    env = PlenVecEnv(n, auto_reset=False, config_overrides={"solver_iterations": its, "residual_threshold": -1.0})
    env.set_state(*abi_from_oracle(o.get_state()))
    env.tick(torch.from_numpy(F["tgt"]).cuda())
    for e in range(n):
        o.tick(e)
    qpos, qvel, _ = (_np(t).astype(np.float64) for t in env.get_state())
    ref = o.get_state()
    dv = np.abs(qvel - ref["qvel"]).max(1)
    dq = np.abs(qpos - ref["qpos"]).max(1)
    assert (_np(env.debug_records())[:, 79] == its).all()
    print("plen_tick vs oracle at %d sweeps: worst robot velocity %.2e, pose %.2e" % (its, dv.max(), dq.max()))
    assert dv.max() < ORACLE_BOUND[its][0] and dq.max() < ORACLE_BOUND[its][1]
