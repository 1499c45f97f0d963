"""CPU tests of the per-robot command latency (plen_set_env_latency) through the warp-emulation harness (tests/emu/emu_latency.cpp):
the device selection function against the numpy schedule, and an emulated latency step (k_dyn's latency prologue, the ticks,
env_post) against the stock ticks driven one by one with the scheduled targets."""
import numpy as np

from emu_latency_util import EmuLatency
from latency_util import CommandSchedule, latency_source


def test_selection_function_matches_numpy_schedule():
    emu = EmuLatency()
    for S in (1, 2, 4):
        for d in range(2 * S + 1):
            for k in range(S):
                for ep_t in range(4):
                    got = emu.latency_source(d, k, S, ep_t)
                    assert got == int(latency_source(d, k, S, ep_t)), (S, d, k, ep_t)
                    assert got in (-1, 0, 1, 2)
        # the documented corner cases: d = 0 is the stock path, d = S holds the previous step's command for the whole step
        assert all(emu.latency_source(0, k, S, 0) == 0 for k in range(S))
        assert all(emu.latency_source(S, k, S, 5) == 1 for k in range(S))
        assert all(emu.latency_source(S, k, S, 0) == -1 for k in range(S))
    for ep_t in range(7):
        for s in range(3):
            if s <= ep_t:
                assert emu.latency_slot(ep_t, s) == (ep_t - s) % 3
    # the row tick 0 writes is never one a tick of the same step reads
    assert all(emu.latency_slot(e, 0) not in (emu.latency_slot(e, 1), emu.latency_slot(e, 2)) for e in range(2, 9))


def _snapshot(emu):
    rec = emu.init_record(1)
    emu.tick(rec, np.zeros((1, 18)), int(emu.cfg.reset_ticks))
    return np.concatenate([rec[0], emu.observe(rec)[0]]).astype(np.float32)


def _agent_target(cfg, a):
    """agent_to_env in float64 then float32, as agent_target (plen_env.cuh) computes it."""
    lo, hi = np.array(list(cfg.env_lo)), np.array(list(cfg.env_hi))
    mm = (hi - lo) / 2.0
    y = mm * np.asarray(a, dtype=np.float32).astype(np.float64) + (hi - mm * 1.0)
    y = np.where(y >= hi, hi - 0.001, np.where(y <= lo, lo + 0.001, y))
    return y.astype(np.float32)


def test_latency_step_matches_stock_ticks_with_scheduled_targets():
    """Nine robots with delays 0..8 ticks, switched on mid-episode (the history seeded with their last targets), a reset of
    three robots mid-run and new delays from the sixth step on: every step's records, observations, rewards and done flags are
    bit-identical to emu_tick driven tick by tick with the numpy-scheduled targets, followed by env_post."""
    emu = EmuLatency()
    snap = _snapshot(emu)
    n, S = 9, int(emu.cfg.substeps)
    rng = np.random.default_rng(3)
    rec = np.repeat(snap[None, :96], n, 0).copy()
    # three stock steps first: the robots are mid-episode (ep_t = 3) when the latency is switched on
    for _ in range(3):
        a = rng.uniform(-0.4, 0.4, (n, 18)).astype(np.float32)
        emu.step(rec, a, snap)
    last = _agent_target(emu.cfg, a)
    assert (rec[:, 63] == 3).all()
    ref = rec.copy()
    ring = emu.new_ring(last)
    sched = CommandSchedule(n, S, last)
    d = np.arange(n, dtype=np.int32)
    differs = 0
    for t in range(10):
        if t == 4:      # explicit reset of three robots, mirrored in the reference
            m = np.array([1, 4, 8])
            rec[m] = snap[:96]
            ref[m] = snap[:96]
        if t == 6:      # new delays between two steps
            d = rng.permutation(n).astype(np.int32)
        a = rng.uniform(-0.4, 0.4, (n, 18)).astype(np.float32)
        raw = _agent_target(emu.cfg, a)
        targets = sched.step(raw, d, ref[:, 63].astype(np.int64))
        obs, rew, done, tgt = emu.step_latency(rec, a, ring, d, snap)
        assert (tgt == raw).all()
        for k in range(S):
            emu.tick(ref, targets[k], 1)
        robs, rrew, rdone = emu.post(ref, snap)
        assert (rec.view(np.uint32) == ref.view(np.uint32)).all(), t
        assert (obs.view(np.uint32) == robs.view(np.uint32)).all(), t
        assert (rew.view(np.uint32) == rrew.view(np.uint32)).all() and (done == rdone).all(), t
        differs += int((targets != raw[None]).any(axis=(0, 2)).sum())
    # the delays did act: robots with d > 0 were driven by targets other than their current command
    assert differs >= 40
