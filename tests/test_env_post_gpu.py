"""GPU tests of k_post (env_post in plen_env.cuh), the env epilogue of every step, robot by robot against float64 references
on constructed states.

With plen_config.substeps = 0 a plen_step runs no physics tick: it is k_post alone on the records the test wrote with
set_state.  The tests call lib.plen_step with their own output buffers, filled with sentinels before each call (a NaN with a
payload the kernel never produces for obs, reward and terminal_obs, 0xAB for done and timeout), so they also see which words
k_post writes.  References: the float64 build of the device source (tests/emu/emu_warp.cpp) and PlenOracle.step at
substeps = 0; the families and the checks are shared with tests/test_env_post_emu.py (tests/env_post_util.py).

Bounds are per robot, never quantiles; robots whose float64 decisive quantity lies within 2e-5 (relative) of a decision
threshold are left out of the checks that depend on it.  The bounds are a few times the worst cases of the float32 build of the
same source on the host (tests/test_env_post_emu.py); they have not yet been measured on a B200."""
import ctypes as C

import numpy as np
import pytest
import torch

import env_post_util as U
from emu_util import Emu

pytestmark = pytest.mark.gpu

REWARD_REL = 1e-5                 # reward within 1e-5 max(1, |r|) of both references
EULER = 2e-6                      # Euler angles, plus 2e-7 / cos(pitch) towards the gimbal cut (env_post_util.euler_bound)
SUMS_REL = 1e-6                   # history sums, relative to the larger of the old and the new sum
SENT_F = np.uint32(0xFFC0BAAD)    # quiet NaN with a payload: the kernel's own NaNs (0 / 0) are canonical
SENT_B = 0xAB


@pytest.fixture(scope="module")
def fam(oracle_lib):
    rec, labels, names = U.all_families(seed=0)
    q = U.quantities(rec)
    e64 = Emu(double=True)
    out = dict(rec=rec, labels=labels, names=names, q=q, fault=U.faulted(rec), near=U.near_threshold(q),
               e64=U.emu_post(e64, rec, U.snapshot_record(e64)), orc=U.oracle_post(rec))
    out["counts"] = U.branch_counts(rec, q, out["orc"]["reward"])
    U.check_coverage(out["counts"])
    return out


def _env(n, auto_reset=False, **cfg):
    from plen_ml_walk_b200.vec_env import PlenVecEnv
    return PlenVecEnv(n, auto_reset=auto_reset, config_overrides=dict(substeps=0, **cfg))


def _load(env, rec):
    env.set_state(*U.record_to_state(rec))


def _sentinel_f(shape):
    return torch.from_numpy(np.full(shape, SENT_F, np.uint32).view(np.float32)).cuda()


def _bufs(n):
    return dict(obs=_sentinel_f((n, 26)), reward=_sentinel_f((n,)), terminal_obs=_sentinel_f((n, 26)),
                done=torch.full((n,), SENT_B, dtype=torch.uint8, device="cuda"),
                timeout=torch.full((n,), SENT_B, dtype=torch.uint8, device="cuda"))


def _out(b, rec):
    o = {k: v.cpu().numpy() for k, v in b.items()}
    o["rec"] = rec
    return o


def _step(env, lib=None, ctx=None):
    """one plen_step with fresh sentinel buffers -> dict of numpy outputs and the records after it"""
    lib, ctx = (env.lib, env._ctx) if env is not None else (lib, ctx)
    n = lib.plen_num_envs(ctx)
    b = _bufs(n)
    act = torch.zeros((n, 18), dtype=torch.float32, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    assert lib.plen_step(ctx, p(act), p(b["obs"]), p(b["reward"]), p(b["done"]), p(b["timeout"]), p(b["terminal_obs"]),
                         C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
    torch.cuda.synchronize()
    return _out(b, env.debug_records().cpu().numpy() if env is not None else None)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _snapshot(env):
    """the post-reset record, observation and manifolds of a fresh context (every robot holds them after plen_create)"""
    rec = env.debug_records().cpu().numpy()[0].copy()
    obs = env.reset().cpu().numpy()[0].copy()
    man = env.get_manifold().cpu().numpy()[0].copy() if env.cfg.sole_manifold else None
    return rec, obs, man


def _as64(o):
    return dict(o, obs=o["obs"].astype(np.float64), reward=o["reward"].astype(np.float64), rec=o["rec"].astype(np.float64))


@pytest.fixture(scope="module")
def run(fam):
    """the families through k_post once, auto-reset off; the snapshot and the fault counter around the step"""
    rec = fam["rec"]
    env = _env(rec.shape[0])
    try:
        snap = _snapshot(env)
        f0 = env.fault_count()
        _load(env, rec)
        out = _step(env)
        f1 = env.fault_count()
    finally:
        env.close()
    return dict(out=out, snap=snap, faults=f1 - f0)


def test_k_post_writes_every_output(fam, run):
    """every output slot is written for every robot; terminal_obs exactly where done is set"""
    o = run["out"]
    assert not (_bits(o["obs"]) == SENT_F).any() and not (_bits(o["reward"]) == SENT_F).any()
    assert np.isin(o["done"], (0, 1)).all() and np.isin(o["timeout"], (0, 1)).all()
    t = _bits(o["terminal_obs"]) == SENT_F
    d = o["done"] == 1
    assert t[~d].all() and not t[d].any()
    # without auto-reset the terminal observation of a robot that is not faulted is its observation
    k = d & ~fam["fault"]
    assert np.array_equal(_bits(o["terminal_obs"][k]), _bits(o["obs"][k]))


@pytest.mark.parametrize("ref", ["e64", "orc"])
def test_k_post_against_float64(fam, run, ref):
    """observation (copied words bit for bit, Euler angles within 2e-6), counters, last, done, timeout exact; reward NaN
    pattern exact; reward within 1e-5 max(1, |r|); sums within 1e-6; ep_ret within the reward bound plus 1 ulp"""
    rec, q, near = fam["rec"], fam["q"], fam["near"]
    ok = ~fam["fault"]
    for f in U.FAMILIES:
        m = fam["names"] == f
        print("%s: %d robots, %d left out of the decision checks (near a threshold)" % (f, m.sum(), (near & m).sum()))
        assert (near & m).sum() <= 0.05 * m.sum(), f
    got = _as64(run["out"])
    mism = U.step_mismatches(got, fam[ref], rec, ok, near, REWARD_REL, U.euler_bound(q, EULER), SUMS_REL)
    U.report(mism, fam["labels"], "k_post vs %s" % ref)
    r = fam[ref]
    with np.errstate(invalid="ignore"):
        dr = np.abs(got["reward"] - r["reward"]) / np.maximum(1.0, np.abs(r["reward"]))
        de = np.abs(got["obs"][:, 20:23] - r["obs"][:, 20:23]).max(1)
        s1 = r["rec"][:, U.W_SUMS:U.W_SUMS + 9]
        ds = (np.abs(got["rec"][:, U.W_SUMS:U.W_SUMS + 9] - s1) /
              np.maximum(np.maximum(np.abs(rec[:, U.W_SUMS:U.W_SUMS + 9]), np.abs(s1)), 1e-300)).max(1)
    k = ok & ~near
    reg = k & (np.abs(q["sarg"]) < 0.9999)
    print("worst vs %s: reward %.3g, Euler %.3g (%.3g away from the gimbal cut), sums %.3g" %
          (ref, np.nanmax(dr[k]), np.nanmax(de[k]), np.nanmax(de[reg]), np.nanmax(ds[ok])))


def test_k_post_numeric_guard(fam, run):
    """faulted robots are reset with auto-reset off: reward exactly -100, done 1, timeout 0 (also at ept = max - 1), record
    and observation from the snapshot, terminal_obs the snapshot observation; fault_count rises by their number"""
    o, (srec, sobs, _) = run["out"], run["snap"]
    f = fam["fault"]
    assert (o["reward"][f] == -100.0).all() and (o["done"][f] == 1).all() and (o["timeout"][f] == 0).all()
    assert (_bits(o["rec"][f]) == _bits(srec)).all()
    assert (_bits(o["obs"][f]) == _bits(sobs)).all() and (_bits(o["terminal_obs"][f]) == _bits(sobs)).all()
    assert run["faults"] == f.sum()
    lam = np.isnan(fam["rec"][:, U.W_LAM:U.W_LAM + 8]).any(1)        # NaN impulses alone: no fault, the NaN words stay
    assert np.array_equal(np.isnan(o["rec"][lam, U.W_LAM:U.W_LAM + 8]), np.isnan(fam["rec"][lam, U.W_LAM:U.W_LAM + 8]))


def test_k_post_leaves_other_words(fam):
    """through the tick harness, whose state view holds all 96 words: the words env_post neither reads nor writes (37, W_ITERS,
    80-95) come back bit-identical for every robot that is not reset, and a faulted robot is the snapshot record"""
    from tick_harness_util import TickCtx
    rng = np.random.default_rng(5)
    rec = fam["rec"].copy()
    rec[:, U.UNTOUCHED] = rng.standard_normal((rec.shape[0], len(U.UNTOUCHED))).astype(np.float32)
    ctx = TickCtx(rec.shape[0], {"substeps": 0})
    try:
        snap = ctx.state[0].cpu().numpy().copy()
        ctx.state.copy_(torch.from_numpy(rec).cuda())
        ctx.L.plen_step.argtypes = [C.c_void_p] * 8
        ctx.L.plen_num_envs.argtypes = [C.c_void_p]
        _step(None, ctx.L, ctx.ctx)
        after = ctx.state.cpu().numpy()
    finally:
        ctx.close()
    f = fam["fault"]
    assert np.array_equal(_bits(after[~f][:, U.UNTOUCHED]), _bits(rec[~f][:, U.UNTOUCHED]))
    assert (_bits(after[f]) == _bits(snap)).all()


def test_k_post_auto_reset(fam):
    """the same records through auto_reset = 1 and auto_reset = 0 contexts with persistent sole manifolds: reward, done and
    timeout bit-identical; a done robot holds the snapshot's record and manifolds, the reset observation and, as terminal_obs,
    the auto_reset = 0 observation; robots that are not done are bit-identical between the two and keep their manifolds"""
    rec = fam["rec"]
    n = rec.shape[0]
    garbage = torch.from_numpy(np.random.default_rng(6).standard_normal((n, 52)).astype(np.float32)).cuda()
    outs, mans = [], []
    for ar in (1, 0):
        env = _env(n, auto_reset=bool(ar), sole_manifold=1)
        try:
            if ar:
                srec, sobs, sman = _snapshot(env)
            _load(env, rec)
            env.set_manifold(garbage)
            outs.append(_step(env))
            mans.append(env.get_manifold().cpu().numpy())
        finally:
            env.close()
    a, b = outs
    g = garbage.cpu().numpy()
    for k in ("reward", "done", "timeout"):
        assert np.array_equal(_bits(a[k]) if a[k].dtype == np.float32 else a[k], _bits(b[k]) if b[k].dtype == np.float32 else b[k]), k
    d = a["done"] == 1
    f = fam["fault"]
    assert d.sum() > 100 and (~d).sum() > 100
    assert (_bits(a["rec"][d]) == _bits(srec)).all() and (_bits(a["obs"][d]) == _bits(sobs)).all()
    assert np.array_equal(_bits(a["terminal_obs"][d]), _bits(b["obs"][d]))
    assert (_bits(mans[0][d]) == _bits(sman)).all() and np.array_equal(_bits(mans[0][~d]), _bits(g[~d]))
    assert (_bits(mans[1][f]) == _bits(sman)).all() and np.array_equal(_bits(mans[1][~f]), _bits(g[~f]))
    assert np.array_equal(_bits(a["rec"][~d]), _bits(b["rec"][~d])) and np.array_equal(_bits(a["obs"][~d]), _bits(b["obs"][~d]))


def test_k_post_time_limit_over_steps():
    """max_episode_steps = 3, auto-reset on, 10 steps: robots that never die time out at steps 3, 6 and 9 with ept and ep_ret
    restarting from the snapshot; a robot in a dead pose at ept = 2 reports done 1, timeout 0 on its timeout step, then
    times out at steps 4, 7 and 10"""
    n = 64
    env = _env(n, auto_reset=True, max_episode_steps=3)
    try:
        srec, _, _ = _snapshot(env)
        rec = np.tile(srec, (n, 1))
        dying = np.arange(n) % 2 == 1
        rec[dying, U.W_POS + 2] = 0.05
        rec[dying, U.W_EPT] = 2
        _load(env, rec)
        ept, ret = np.where(dying, 2, 0), np.zeros(n, np.float32)
        for t in range(1, 11):
            o = _step(env)
            exp_done = np.where(dying, t % 3 == 1, t % 3 == 0)
            exp_tmo = exp_done & ~(dying & (t == 1))
            assert np.array_equal(o["done"] == 1, exp_done), t
            assert np.array_equal(o["timeout"] == 1, exp_tmo), t
            ret = np.where(exp_done, np.float32(0), ret + o["reward"]).astype(np.float32)
            ept = np.where(exp_done, 0, ept + 1)
            assert np.array_equal(o["rec"][:, U.W_EPT], ept), t
            assert np.array_equal(_bits(o["rec"][:, U.W_EPRET]), _bits(ret)), t
    finally:
        env.close()


def test_k_post_launch_geometry(fam):
    """all families mixed, permuted, at n = 1, 37 (not a multiple of the 10 warps per CTA), 2,085 (the two fanned-out ranges of
    plen_step), 9,000 and 40,000 (2 and 4 ranges of plen_step_host): every robot's outputs and record are bit-identical to its
    own in the whole-family run, whatever its position, the batch size and the entry point (plen_step_host: no terminal_obs)"""
    rec = fam["rec"]
    N = rec.shape[0]
    env = _env(N, auto_reset=True)
    try:
        _load(env, rec)
        base = _step(env)
    finally:
        env.close()
    rng = np.random.default_rng(7)
    for n in (1, 37, 2085, 9000, 40000):
        idx = np.concatenate([rng.permutation(N) for _ in range(n // N + 1)])[:n]
        env = _env(n, auto_reset=True)
        try:
            _load(env, rec[idx])
            o = _step(env)
            for k in ("obs", "reward", "done", "timeout", "terminal_obs", "rec"):
                a, b = o[k], base[k][idx]
                if a.dtype == np.float32:
                    a, b = _bits(a), _bits(b)
                assert np.array_equal(a, b), (n, k, fam["labels"][idx][np.where((a != b).reshape(n, -1).any(1))[0][:4]])
            if n >= 9000:
                _load(env, rec[idx])
                h = dict(obs=np.full((n, 26), SENT_F, np.uint32).view(np.float32), reward=np.full(n, SENT_F, np.uint32).view(np.float32),
                         done=np.full(n, SENT_B, np.uint8), timeout=np.full(n, SENT_B, np.uint8))
                env.step_host(np.zeros((n, 18), np.float32), h["obs"], h["reward"], h["done"], h["timeout"])
                h["rec"] = env.debug_records().cpu().numpy()
                for k in ("obs", "reward", "done", "timeout", "rec"):
                    a, b = h[k], base[k][idx]
                    if a.dtype == np.float32:
                        a, b = _bits(a), _bits(b)
                    assert np.array_equal(a, b), ("step_host", n, k)
        finally:
            env.close()


def test_plen_reset_masked(fam):
    """plen_reset with a mask restores the record and manifolds of the masked robots only, writes their observation only and
    leaves the other robots' observation sentinels in place"""
    rec = fam["rec"][:300]
    n = rec.shape[0]
    env = _env(n, sole_manifold=1)
    try:
        srec, sobs, sman = _snapshot(env)
        _load(env, rec)
        garbage = torch.from_numpy(np.random.default_rng(8).standard_normal((n, 52)).astype(np.float32)).cuda()
        env.set_manifold(garbage)
        before = env.debug_records().cpu().numpy()
        mask = torch.from_numpy(np.random.default_rng(9).random(n) < 0.5).to(torch.uint8).cuda()
        obs = _sentinel_f((n, 26))
        assert env.lib.plen_reset(env._ctx, C.c_void_p(mask.data_ptr()), C.c_void_p(obs.data_ptr()), env._stream()) == 0
        torch.cuda.synchronize()
        after, man, obs = env.debug_records().cpu().numpy(), env.get_manifold().cpu().numpy(), obs.cpu().numpy()
    finally:
        env.close()
    m = mask.cpu().numpy() == 1
    g = garbage.cpu().numpy()
    assert 50 < m.sum() < n - 50
    assert (_bits(after[m]) == _bits(srec)).all() and (_bits(man[m]) == _bits(sman)).all() and (_bits(obs[m]) == _bits(sobs)).all()
    assert np.array_equal(_bits(after[~m]), _bits(before[~m])) and np.array_equal(_bits(man[~m]), _bits(g[~m]))
    assert (_bits(obs[~m]) == SENT_F).all()
