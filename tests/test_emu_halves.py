"""CPU tests of the two halves of a physics tick in the warp emulation (tests/emu/emu_halves.cpp): k_dyn's solve record and
k_solve's projected Gauss-Seidel (PGS), each on its own, in float32 and float64.

These are the references of the GPU tests in tests/test_tick_halves_gpu.py, which run the same halves on the sm_100a build:
the halves must compose to the emulated tick bit for bit, and the float32 source must stay close enough to the float64 one
that the GPU's bounds can be a few times the float32 error.  PGS capped at k sweeps with the early exit off
(residual_threshold < 0) is a composition of continuous piecewise-linear clamps, so its float32 and float64 results agree
tightly; the stock 50 sweeps amplify round-off chaotically at impacts (DESIGN.md section 1, 'PGS sensitivity')."""
import os

import numpy as np
import pytest

from emu_halves_util import SR_MAN, SWEEP_BOUND, XR_NX, EmuHalves, ext_errors, make_family, record_errors, sort_keys
from emu_util import oracle_state_from_record


@pytest.fixture(scope="module")
def emus():
    return EmuHalves(), EmuHalves(double=True)


def test_tick_harness_compiles_and_loads():
    """tests/cuda/tick_harness.cu includes plen_b200.cu: it must keep compiling for sm_100a and load without undefined
    symbols, or the GPU tests of the tick halves would break unnoticed when the library's sources change."""
    import ctypes
    import tick_harness_util
    if not os.path.exists(tick_harness_util.nvcc()):
        pytest.skip("nvcc not available")
    lib = ctypes.CDLL(tick_harness_util.build_harness())
    for sym in ("th_buffers", "th_sizes", "th_dyn", "th_rank", "th_solve", "th_set_solver", "plen_create", "plen_tick"):
        assert getattr(lib, sym)
    sizes = (ctypes.c_int * 8)()
    assert lib.th_sizes(sizes) == 8
    assert list(sizes) == [1600, 976, 125, 128, 160, 1024, 8, 32]


@pytest.mark.parametrize("double", [False, True])
@pytest.mark.parametrize("mass", [False, True])
def test_halves_compose_to_emu_tick(oracle_lib, double, mass):
    """emu_dyn then emu_solve is emu_tick (emu_tick_mass with mass rows) bit for bit: the halves the GPU tests compare
    against are the emulated tick, not a re-implementation of it.  Contact states and fallen poses (box contacts), 40 robots:
    five solver groups, two of them EXT."""
    from emu_mass_util import EmuMass, mass_rows
    h = EmuHalves(double=double)
    ref = EmuMass(double=double)
    fa, fb = make_family(oracle_lib, "contact", 24, seed=1), make_family(oracle_lib, "fallen", 16, seed=2)
    rec = np.concatenate([fa["rec"], fb["rec"]]).astype(h.real)
    tg = np.concatenate([fa["tgt"], fb["tgt"]])
    n = rec.shape[0]
    rows = None
    if mass:
        rng = np.random.default_rng(3)
        pay = np.zeros((n, 4))
        pay[:, 0] = rng.uniform(0, 0.1, n)
        rows = mass_rows(rng.uniform(0.8, 1.3, (n, 19)), pay, dtype=h.real)
        ref.set_mass(rows)
    r1 = rec.copy()
    ref.tick(r1, tg, 1)
    r2 = rec.copy()
    srec, srx, keys = h.dyn(r2, tg, mass_rows=rows)
    assert (keys >= 125).sum() >= 8 and (keys < 125).sum() >= 8
    h.solve(r2, srec, srx, keys)
    assert np.array_equal(r1, r2)


def test_f32_vs_f64_records_and_capped_sweeps(oracle_lib, emus):
    """Same float32 state, float32 against float64 evaluation of the same device source:
      - k_dyn: keys, manifold bits and box point counts identical; every solve-record element within 5e-4 of its row's block
        maximum (a 32-word row of G or B, the whole block elsewhere; measured worst case 1.3e-4, in B); the box-contact
        rows part by part likewise (measured 1.9e-5).
      - k_solve on the float32 record, capped at k = 1, 2, 4, 8 sweeps without early exit: every robot's velocities within
        SWEEP_BOUND[k] rad/s or m/s (measured worst cases 1.6e-4, 7.8e-5, 2.9e-4, 1.4e-3 over two sets of states: each
        sweep re-decides the clamps of the box lateral pairs, so the error grows with k), the iteration word exact."""
    e32, e64 = emus
    fams = [make_family(oracle_lib, f, 32, seed=10 + i) for i, f in enumerate(("contact", "fallen", "limits"))]
    rec = np.concatenate([f["rec"] for f in fams])
    tg = np.concatenate([f["tgt"] for f in fams])
    s32, x32, k32 = e32.dyn(rec, tg)
    s64, x64, k64 = e64.dyn(rec, tg)
    assert np.array_equal(k32, k64) and np.array_equal(s32[:, SR_MAN], s64[:, SR_MAN])
    assert np.array_equal(k32, sort_keys(s32, x32)) and np.array_equal(x32[:, XR_NX], x64[:, XR_NX])
    worst = {k: v.max() for k, v in record_errors(s32, s64).items()}
    xw = {k: v.max() for k, v in ext_errors(x32, x64).items()}
    xr = max(xw.values())
    print("record f32 vs f64, rel. to block max:", {k: "%.1e" % v for k, v in worst.items()}, {k: "%.1e" % v for k, v in xw.items()})
    assert max(worst.values()) < 5e-4 and xr < 5e-4
    errs = {}
    try:
        for its in (1, 2, 4, 8):
            e32.set_solver(its, -1.0)
            e64.set_solver(its, -1.0)
            ra, rb = rec.copy(), rec.astype(np.float64)
            e32.solve(ra, s32, x32, k32)
            e64.solve(rb, s32, x32, k32)
            errs[its] = np.abs(ra[:, :24] - rb[:, :24]).max(1)
            assert (ra[:, 79] == its).all() and (rb[:, 79] == its).all()
    finally:
        e32.set_solver(50, 1e-7)
        e64.set_solver(50, 1e-7)
    print("capped sweeps f32 vs f64 solve, worst robot:", {k: "%.1e" % v.max() for k, v in errs.items()})
    for its, v in errs.items():
        assert v.max() < SWEEP_BOUND[its]


@pytest.mark.parametrize("its", [1, 4])
def test_f64_emulation_vs_oracle_capped_sweeps(oracle_lib, its):
    """One tick from oracle states (contact, fallen poses with box contacts, limit rows) in the float64 emulation against
    PlenOracle.tick, both capped at `its` sweeps with the early exit off.  The same algorithm in float64 (the model tables
    stay float32) must agree per robot to 1.5e-4 rad/s or m/s in velocity and 6e-7 in pose (measured worst cases 4.5e-5 and
    1.9e-7 at 1 sweep, 3.7e-5 and 1.6e-7 at 4 sweeps): no quantile, no excluded robot.  The counterpart of the GPU leg
    test_whole_tick_vs_oracle_capped_sweeps."""
    e64 = EmuHalves(double=True)
    e64.set_solver(its, -1.0)
    fams = [make_family(oracle_lib, f, 16, seed=20 + i) for i, f in enumerate(("contact", "fallen", "limits"))]
    rec = np.concatenate([f["rec"] for f in fams]).astype(np.float64)
    tg = np.concatenate([f["tgt"] for f in fams]).astype(np.float64)
    n = rec.shape[0]
    o = oracle_lib.PlenOracle(n)
    o.cfg.solver_iterations = its
    o.cfg.residual_threshold = -1.0
    st = oracle_state_from_record(rec)
    st["target"] = tg
    o.set_state(st)
    srec, srx, keys = e64.dyn(rec, tg)
    assert (keys >= 125).sum() >= 8
    e64.solve(rec, srec, srx, keys)
    for e in range(n):
        o.tick(e)
    got, ref = oracle_state_from_record(rec), o.get_state()
    dv = np.abs(got["qvel"] - ref["qvel"]).max(1)
    dq = np.abs(got["qpos"] - ref["qpos"]).max(1)
    assert all(o.states[e].last_iterations == its for e in range(n))
    print("f64 emulation vs oracle at %d sweeps: worst robot velocity %.1e, pose %.1e" % (its, dv.max(), dq.max()))
    assert dv.max() < 1.5e-4 and dq.max() < 6e-7
