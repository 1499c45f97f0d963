"""CPU tests of env_post (plen_env.cuh), the env epilogue of a step, on constructed states: the warp emulation of the device
source at substeps = 0, where a step is env_post alone, against PlenOracle.step at substeps = 0 on the same records.

The families (tests/env_post_util.py) put a few hundred labelled robots on each branch: every gait-schedule counter edge,
double support, degenerate history sums, termination and gimbal thresholds, foot flatness, vx signs, TimeLimit and the
numeric guard.  Every test checks that each branch is still taken by at least 8 robots."""
import numpy as np
import pytest

import env_post_util as U
from emu_util import Emu

# float64 emulation against the oracle, both float64 on the same float32 records.  The reward differs only through the float32
# literal 0.160178937611f of the height term, 6.9e-9 m off the reference constant: d(h^2) = 2 |h| 40 * 6.9e-9, 1.2e-6 at
# |h| = 2.1 (worst measured 7.9e-7 over these families).  The gimbal pitch is the float32 literal 1.57079632679f, 4.4e-8 off
# pi/2; every other observation word is exact.
ORACLE_REWARD_REL = 5e-6
GIMBAL_PITCH_LITERAL = 5e-8
# the float32 literals of pi/3, 0.08, 0.1 and 0.99999 lie within 3e-8 (relative) of the reference's thresholds
LITERAL_REL = 1e-7
# float32 emulation against float64 (measured: reward 1.6e-6, sums 7.2e-7 of the larger of the old and new sum, Euler angles
# 2.3e-7 away from the gimbal cut and 5.0e-6 at sarg = -0.99994, see env_post_util.euler_bound)
F32_REWARD_REL = 5e-6
F32_SUMS_REL = 2e-6
F32_EULER = 2e-6


@pytest.fixture(scope="module")
def fam(oracle_lib):
    rec, labels, names = U.all_families(seed=0)
    q = U.quantities(rec)
    e64, e32 = Emu(double=True), Emu()
    s64, s32 = U.snapshot_record(e64), U.snapshot_record(e32)
    out = dict(rec=rec, labels=labels, names=names, q=q, fault=U.faulted(rec), near=U.near_threshold(q),
               e64=U.emu_post(e64, rec, s64), e32=U.emu_post(e32, rec, s32), orc=U.oracle_post(rec), s64=s64, s32=s32)
    out["e64_auto"] = U.emu_post(e64, rec, s64, auto_reset=1)
    U.check_coverage(U.branch_counts(rec, q, out["orc"]["reward"]))
    return out


def test_families_cover_every_branch(fam):
    """each family keeps its point: the float64 reference takes every branch of env_post at least 8 times, and at most 5 % of
    any family lies within 2e-5 of a decision threshold (those robots are left out of the float32 decision checks)"""
    for f in U.FAMILIES:
        m = fam["names"] == f
        print("%s: %d robots, %d near a threshold" % (f, m.sum(), (fam["near"] & m).sum()))
        assert (fam["near"] & m).sum() <= 0.05 * m.sum(), f
    assert fam["fault"].sum() == 3 * (24 + 18 + 3 + 4)


def test_emu_f64_matches_oracle(fam):
    """the float64 build of the device source against PlenOracle.step, robot by robot: observation exact (gimbal pitch: the
    float32 literal of pi/2), counters and last exact, reward NaN pattern, done and timeout exact, reward within 5e-6"""
    rec, q = fam["rec"], fam["q"]
    eb = np.zeros((rec.shape[0], 3))
    eb[np.abs(q["sarg"]) >= U.SARG_GIMBAL, 1] = GIMBAL_PITCH_LITERAL
    ok = ~fam["fault"]
    m = U.step_mismatches(fam["e64"], fam["orc"], rec, ok, U.near_threshold(q, LITERAL_REL), ORACLE_REWARD_REL, eb, 0.0)
    U.report(m, fam["labels"], "float64 emulation vs oracle")
    words = [k for k in range(26) if k not in (20, 21, 22)]
    assert np.array_equal(fam["e64"]["obs"][ok][:, words], fam["orc"]["obs"][ok][:, words])
    with np.errstate(invalid="ignore"):
        d = np.abs(fam["e64"]["reward"] - fam["orc"]["reward"]) / np.maximum(1.0, np.abs(fam["orc"]["reward"]))
    print("worst reward difference %.3g" % np.nanmax(d[ok]))


def test_emu_f32_matches_f64(fam):
    """the float32 emulation against the float64 one on the same records, robots near a decision threshold left out of the
    decision checks"""
    rec, q = fam["rec"], fam["q"]
    ok = ~fam["fault"]
    m = U.step_mismatches(fam["e32"], fam["e64"], rec, ok, fam["near"], F32_REWARD_REL, U.euler_bound(q, F32_EULER), F32_SUMS_REL)
    U.report(m, fam["labels"], "float32 vs float64 emulation")


@pytest.mark.parametrize("prec", ["e64", "e32"])
def test_emu_numeric_guard(fam, prec):
    """a non-finite velocity, joint angle, position or quaternion word retires the robot with auto-reset off: reward exactly
    -100, done 1, timeout 0 (also at ept = max - 1), record, observation and terminal observation from the snapshot.  NaN in
    the cached normal impulses alone is no fault: that robot steps as usual and keeps its NaN words."""
    out, s = fam[prec], fam["s64" if prec == "e64" else "s32"]
    f = fam["fault"]
    assert (out["reward"][f] == -100.0).all() and out["done"][f].all() and not out["timeout"][f].any()
    assert (out["rec"][f] == s[:96].astype(np.float64)).all()
    assert (out["obs"][f] == s[96:].astype(np.float64)).all() and (out["terminal_obs"][f] == s[96:].astype(np.float64)).all()
    lam = np.isnan(fam["rec"][:, U.W_LAM:U.W_LAM + 8]).any(1)
    assert lam.sum() == 24 and not (f & lam).any()
    assert np.array_equal(np.isnan(out["rec"][lam, U.W_LAM:U.W_LAM + 8]), np.isnan(fam["rec"][lam, U.W_LAM:U.W_LAM + 8]))
    assert np.array_equal(out["done"][lam], fam["orc"]["done"][lam])


def test_emu_auto_reset(fam):
    """auto_reset = 1 against auto_reset = 0 on the same records: identical reward, done and timeout; a done robot is the
    snapshot's record and observation with the auto_reset = 0 observation as its terminal observation; the others step alike"""
    a, b, s = fam["e64_auto"], fam["e64"], fam["s64"]
    assert np.array_equal(a["reward"], b["reward"], equal_nan=True)
    assert np.array_equal(a["done"], b["done"]) and np.array_equal(a["timeout"], b["timeout"])
    d = a["done"]
    assert d.sum() > 100 and (~d).sum() > 100
    assert (a["rec"][d] == s[:96]).all() and (a["obs"][d] == s[96:]).all()
    assert np.array_equal(a["terminal_obs"][d], b["obs"][d])
    assert np.array_equal(a["rec"][~d], b["rec"][~d], equal_nan=True) and np.array_equal(a["obs"][~d], b["obs"][~d])
