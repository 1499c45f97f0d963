"""CPU tests of the per-robot reset settle (plen_settle_env_resets) through the warp-emulation harness (tests/emu/emu_resets.cpp):
the device's start_record against a start state built independently, and start_record followed by reset_ticks emulated ticks
against the float64 oracle's reset procedure from the same start poses."""
import numpy as np

from resets_util import EmuResets, oracle_settle, start_qpos

# turned, shifted and raised / lowered starts; the first is the reference's own start (plen_env.py:312)
POSES = np.array([[0.0, 0.0, 0.158, 0.0],
                  [0.0, 0.0, 0.158, 0.3],
                  [0.0, 0.0, 0.158, -0.3],
                  [0.4, -0.25, 0.158, 1.2],
                  [-1.5, 2.0, 0.165, -2.5],
                  [0.1, 0.1, 0.150, 3.1]], dtype=np.float32)


def test_start_record_is_the_teleported_state():
    """Record words: base position, quaternion (0, 0, sin(yaw/2), cos(yaw/2)) and nothing else; yaw 0 is init_record."""
    for double in (False, True):
        emu = EmuResets(double=double)
        rec = emu.start_record(POSES)
        q = start_qpos(POSES)
        assert (rec[:, 32:35] == POSES[:, 0:3]).all()
        if double:      # float64 build: the exact half-angle functions of the float32 yaw
            h = 0.5 * POSES[:, 3].astype(np.float64)
            assert (rec[:, 58] == np.sin(h)).all() and (rec[:, 59] == np.cos(h)).all()
        else:
            assert (rec[:, 56:60] == q[:, 3:7]).all()
        rest = np.delete(rec, [32, 33, 34, 56, 57, 58, 59], axis=1)
        assert (rest == 0).all() and (rec[:, 56:58] == 0).all()
        assert (emu.start_record(POSES[:1]) == emu.init_record(1)).all()


def test_emulated_settle_matches_the_oracle(oracle_lib):
    """start_record + reset_ticks ticks with hold target 0, observed: the float64 build follows the oracle's settle within 1e-6,
    the float32 build within 1e-5 (the bound test_gpu_parity.py holds for the reset from the default pose)."""
    _, ref = oracle_settle(oracle_lib, POSES)
    errs = {}
    for double, bound in ((True, 1e-6), (False, 1e-5)):
        emu = EmuResets(double=double)
        rec, obs = emu.settle(POSES)
        errs[double] = np.abs(obs.astype(np.float64) - ref).max(1)
        assert errs[double].max() < bound, (double, errs[double])
        # the pose did act: headings reach the observed yaw, positions the observed y
        assert np.abs(obs[:, 22] - POSES[:, 3]).max() < 0.05 and np.abs(obs[:, 23] - POSES[:, 1]).max() < 0.01
    print("settle vs oracle: f64 %.2e, f32 %.2e" % (errs[True].max(), errs[False].max()))


def test_emulated_settle_with_sole_manifolds_matches_the_oracle(oracle_lib):
    """The same with the persistent sole manifolds (config sole_manifold = 1, oracle manifold_mode 1), which start empty."""
    o, ref = oracle_settle(oracle_lib, POSES, manifold_mode=1)
    for double, bound in ((True, 1e-6), (False, 1e-5)):
        emu = EmuResets(double=double)
        emu.cfg.sole_manifold = 1
        man = np.zeros((POSES.shape[0], 52), dtype=emu.real)
        emu.set_manifold(man)
        try:
            rec, obs = emu.settle(POSES)
        finally:
            emu.set_manifold(None)
        assert np.abs(obs.astype(np.float64) - ref).max() < bound, double
        assert (man[:, 48:50] == o.get_manifold()[:, 48:50]).all() and (man[:, 48:50].sum(1) > 0).all()
