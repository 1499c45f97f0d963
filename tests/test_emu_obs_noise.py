"""CPU tests of the per-robot observation noise (plen_set_env_obs_noise): the device's generator against the numpy twin
(tests/obs_noise_util.py), and env_post's noise instance through the warp emulation (tests/emu/emu_obs_noise.cpp) on the
constructed families of tests/env_post_util.py at substeps = 0, against env_post's stock instance on the same records."""
import numpy as np
import pytest

import env_post_util as P
import obs_noise_util as U
from emu_util import Emu

# Gaussians of the emulated generator (host libm in double on the float32 uniforms) against the twin's float64 Box-Muller:
# measured worst 4.0e-8 (1 + |n|) over 10^6 keys (the float32 rounding of the result); held to 3x that.  The device's
# logf / cospif add a few float32 ulps more (tests/test_gpu_obs_noise.py holds the GPU to 3.5e-7 (1 + |n|)).
EMU_NORMAL_REL = 1.2e-7
F32_EPS = 2.0 ** -23
SEED = 0x5EED1234ABCD


def _keys(rng, n):
    return rng.integers(0, 2 ** 63, size=n, dtype=np.int64).astype(np.uint64) * np.uint64(2) + rng.integers(0, 2, size=n).astype(np.uint64)


def test_generator_matches_the_twin():
    """hash bits, both float32 uniforms and flip decisions bit for bit over 10^6 keys; p = 0 never flips, p = 1 always; the
    Gaussians within EMU_NORMAL_REL (1 + |n|); the key formula of the header"""
    rng = np.random.default_rng(1)
    e = U.EmuObsNoise()
    k = _keys(rng, 1_000_000)
    p = rng.random(k.size).astype(np.float32)
    p[:1000], p[1000:2000] = 0.0, 1.0
    h, u1, u2, z, f = e.draws(k, p)
    v1, v2 = U.uniforms(k)
    assert (h == U.hash32(k)).all()
    assert (u1.view(np.uint32) == v1.view(np.uint32)).all() and (u2.view(np.uint32) == v2.view(np.uint32)).all()
    assert (f == U.flips(k, p)).all() and not f[:1000].any() and f[1000:2000].all()
    assert (u1 > 0).all() and (u1 <= 1).all() and (u2 >= 0).all() and (u2 < 1).all()
    zt = U.normal(k)
    err = np.abs(z - zt) / (1.0 + np.abs(zt))
    print("emulated Gaussians vs twin: worst %.2e (1 + |n|)" % err.max())
    assert err.max() <= EMU_NORMAL_REL
    for seed, gid, ctr, s, w in ((0, 0, 0, 0, 0), (SEED, 123456, 77, 4, 25), (2 ** 64 - 1, 2 ** 40, 2 ** 32 - 1, 2, 23)):
        assert e.key(seed, gid, ctr, s, w) == int(U.key(seed, np.array([gid]), ctr, s, w)[0])


def _noise_setup(n, rng):
    """per-robot parameters: every 5th word passes through (sigma = beta = 0, b = 0), the rest random; random running biases
    and counters; flip probability 0.3"""
    sigma = rng.uniform(0.0, 0.05, (n, 24)).astype(np.float32)
    beta = rng.uniform(0.0, 0.05, (n, 24)).astype(np.float32)
    bias = rng.normal(0.0, 0.03, (n, 24)).astype(np.float32)
    off = np.zeros(24, bool)
    off[::5] = True
    sigma[:, off] = beta[:, off] = bias[:, off] = 0.0
    ctr = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    return U.rows(n, sigma, beta, 0.3, bias, ctr), off


@pytest.fixture(scope="module", params=[0, 1], ids=["no_auto_reset", "auto_reset"])
def fam(request):
    auto = request.param
    rec, labels, names = P.all_families(seed=0)
    n = rec.shape[0]
    rec = rec.copy()
    rec[::7, P.W_J + 5] = -0.0                     # a -0.0 joint angle (obs word 5, a pass-through word)
    stock_emu = Emu()
    snap = P.snapshot_record(stock_emu).astype(np.float32)
    snap[96 + 10], snap[96 + 15] = np.float32(-0.0), np.float32(np.nan)     # reset observation words 10, 15 (pass-through)
    stock_emu.cfg.substeps, stock_emu.cfg.auto_reset, stock_emu.cfg.max_episode_steps = 0, auto, P.MAX_EP
    r0 = rec.copy()
    stock = stock_emu.step(r0, np.zeros((n, 18)), snap)
    e = U.EmuObsNoise()
    e.cfg.substeps, e.cfg.auto_reset, e.cfg.max_episode_steps = 0, auto, P.MAX_EP
    rng = np.random.default_rng(3)
    rows, off = _noise_setup(n, rng)
    rows0 = rows.copy()
    gid0 = 1000
    r1 = rec.copy()
    noisy = e.step_noise(r1, np.zeros((n, 18)), snap, rows, SEED, gid0)
    reset = (stock[2] & bool(auto)) | P.faulted(rec)
    return dict(rec=rec, stock=stock, stock_rec=r0, noisy=noisy, noisy_rec=r1, rows0=rows0, rows=rows, off=off, snap=snap,
                reset=reset, gid=gid0 + np.arange(n), auto=auto, labels=labels)


def _same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def test_noise_does_not_feed_back(fam):
    """clean observations, reward, done, timeout and records of the noise instance equal the stock instance bit for bit"""
    obs, rew, done, tmo, tobs = fam["stock"]
    nobs, nrew, ndone, ntmo, ntobs, cobs, ctobs = fam["noisy"]
    assert _same_bits(cobs, obs)
    assert _same_bits(nrew, rew) and (ndone == done).all() and (ntmo == tmo).all()
    assert _same_bits(fam["noisy_rec"], fam["stock_rec"])
    assert _same_bits(ctobs[done], tobs[done])
    assert fam["reset"].sum() > 0 and (~fam["reset"]).sum() > 0


def _check_noisy(got, clean, sigma, bias, p, gid, ctr, stream, what):
    exp, f = U.apply(clean, sigma, bias, p, SEED, gid, ctr, stream)
    z = np.abs(U.normal(U.key(SEED, gid[:, None], ctr.astype(np.uint64)[:, None], stream, np.arange(24)[None, :])))
    tol = sigma * EMU_NORMAL_REL * (1 + z) + 2 * F32_EPS * (np.abs(clean[:, :24]) + sigma * z + np.abs(bias))
    with np.errstate(invalid="ignore"):
        bad = ~(np.abs(got[:, :24] - exp[:, :24]) <= tol) & ~(np.isnan(got[:, :24]) & np.isnan(exp[:, :24]))
    assert not bad.any(), (what, np.argwhere(bad)[:5])
    assert (got[:, 24:] == exp[:, 24:]).all(), what
    return f


def test_noisy_minus_clean_is_bias_plus_sigma_n(fam):
    """robots that are not reset: obs = clean + b + sigma n (stream 0) with the running bias, flags flipped by the twin's
    decisions (stream 1), terminal_obs of done robots the same words; the bias is kept and the counter advances by one"""
    nobs, _, done, _, ntobs, cobs, _ = fam["noisy"]
    rows0, rows = fam["rows0"], fam["rows"]
    keep = ~fam["reset"]
    g, c = fam["gid"][keep], U.counters(rows0)[keep]
    f = _check_noisy(nobs[keep], cobs[keep], rows0[keep, :24], rows0[keep, 48:72], rows0[keep, 72], g, c, U.NS_OBS, "step obs")
    assert 0.2 < f.mean() < 0.4
    assert _same_bits(ntobs[keep & done], nobs[keep & done])
    assert _same_bits(rows[keep, 48:72], rows0[keep, 48:72])
    assert (U.counters(rows) == U.counters(rows0) + np.uint32(1)).all()


def test_resets_redraw_the_bias(fam):
    """reset robots (auto-reset, numeric guard): terminal_obs carries the finished episode's bias (stream 0); the new bias is
    beta n' (stream 2); the reset observation is the snapshot's with the new bias and stream 3 / 4 draws"""
    nobs, _, done, _, ntobs, cobs, ctobs = fam["noisy"]
    rows0, rows, snap = fam["rows0"], fam["rows"], fam["snap"]
    rs = fam["reset"]
    g, c = fam["gid"][rs], U.counters(rows0)[rs]
    _check_noisy(ntobs[rs], ctobs[rs], rows0[rs, :24], rows0[rs, 48:72], rows0[rs, 72], g, c, U.NS_OBS, "terminal obs")
    nb = U.new_bias(rows0[rs, 24:48], SEED, g, c)
    z = np.abs(nb / np.where(rows0[rs, 24:48] > 0, rows0[rs, 24:48], 1))
    assert (np.abs(rows[rs, 48:72] - nb) <= rows0[rs, 24:48] * EMU_NORMAL_REL * (1 + z) + F32_EPS * np.abs(nb)).all()
    assert not _same_bits(rows[rs, 48:72], rows0[rs, 48:72])
    clean = np.broadcast_to(snap[96:122], (rs.sum(), 26))
    assert _same_bits(cobs[rs], clean)
    _check_noisy(nobs[rs], clean, rows0[rs, :24], rows[rs, 48:72], rows0[rs, 72], g, c, U.NS_ROBS, "reset obs")


def test_zero_words_pass_through_bit_for_bit(fam):
    """words with sigma = b = 0 are the clean words bit for bit: -0.0 joint angles and the snapshot's -0.0 and NaN words"""
    nobs, _, _, _, _, cobs, _ = fam["noisy"]
    off = np.where(fam["off"])[0]
    assert _same_bits(nobs[:, off], cobs[:, off])
    assert np.signbit(nobs[::7, 5][~fam["reset"][::7]]).all()
    rs = fam["reset"]
    assert np.signbit(nobs[rs, 10]).all() and np.isnan(nobs[rs, 15]).all()
