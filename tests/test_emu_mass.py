"""CPU tests of the per-robot mass tables (plen_set_env_mass) through the warp-emulation harness (tests/emu/emu_mass.cpp): the
MASS instance of the product's tick_dynamics against the float64 oracle run on an equivalent tree, and unit rows against the
stock instance."""
import numpy as np

from emu_mass_util import EmuMass as Emu, mass_rows
from emu_util import oracle_state_from_record, record_from_oracle_state
from mass_util import equivalent_tree, payload_on_base_axis
from plen_ml_walk_b200.urdf_loader import packaged_model


def _groups(tree):
    """Three parameter groups: every body heavier, random per-body scales with a payload above the base com, a heavy payload
    behind it.  Payloads sit on the base link's principal axes, where the oracle's folded base inertia stays diagonal."""
    rng = np.random.default_rng(21)
    return [(np.full(19, 1.3), np.zeros(4)),
            (rng.uniform(0.7, 1.4, 19), payload_on_base_axis(tree, 0.05, 2, 0.02)),
            (np.ones(19), payload_on_base_axis(tree, 0.1, 0, -0.015))]


def test_f64_emulation_with_mass_rows_matches_oracle_on_equivalent_trees(oracle_lib):
    """Teacher-forced through contact ticks like test_f64_emulation_matches_oracle_through_contacts, with its tolerances: each
    group of robots carries its mass row in the emulation and is checked against an oracle whose tree holds the same masses."""
    from oracle.urdf_tree import load_tree
    tree, links = load_tree(), packaged_model().body_links
    groups, per = _groups(tree), 2
    n, ticks = per * len(groups), 6
    oracles = [oracle_lib.PlenOracle(per, tree=equivalent_tree(tree, links, s, p)) for s, p in groups]
    emu = Emu(double=True)
    rows = mass_rows(np.repeat([s for s, _ in groups], per, 0), np.repeat([p for _, p in groups], per, 0), dtype=np.float64)
    emu.set_mass(rows)
    rng = np.random.default_rng(0)
    for o in oracles:
        o.reset()
        for _ in range(6):
            o.step(rng.uniform(-1, 1, (per, 18)))
    qd_err, q_err, same_iters, max_rows = [], [], [], 0
    try:
        for _ in range(ticks):
            st = [o.get_state() for o in oracles]
            rec = np.stack([record_from_oracle_state(s, e, dtype=np.float64) for s in st for e in range(per)])
            tg = rng.uniform(-1, 1, (n, 18))
            for g, o in enumerate(oracles):
                for e in range(per):
                    for k in range(18):
                        o.states[e].target[k] = tg[g * per + e, k]
            emu.tick(rec, tg, 1)
            for o in oracles:
                for e in range(per):
                    o.tick(e)
            ref = [o.get_state() for o in oracles]
            got = oracle_state_from_record(rec)
            qd_err.append(np.abs(got["qvel"] - np.concatenate([r["qvel"] for r in ref])).max(1))
            q_err.append(np.abs(got["qpos"] - np.concatenate([r["qpos"] for r in ref])).max(1))
            its = np.array([o.states[e].last_iterations for o in oracles for e in range(per)])
            same_iters.append(np.mean(rec[:, 79].astype(int) == its))
            max_rows = max(max_rows, max(o.states[e].last_rows for o in oracles for e in range(per)))
    finally:
        emu.set_mass(None)
    qd, q = np.array(qd_err), np.array(q_err)
    print("mass rows vs equivalent trees: qd err median %.2e p80 %.2e, q err median %.2e, same PGS iterations %.2f"
          % (np.median(qd), np.quantile(qd, 0.8), np.median(q), np.mean(same_iters)))
    assert max_rows > 18                         # contact rows were exercised
    assert np.median(qd) < 2e-5 and np.quantile(qd, 0.8) < 1e-3
    assert np.median(q) < 1e-6
    assert np.mean(same_iters) > 0.9


def test_f64_equivalent_tree_differs_from_stock(oracle_lib):
    """The check above has teeth: the stock oracle, stepped from the same states, is far from the mass-row emulation."""
    from oracle.urdf_tree import load_tree
    tree, links = load_tree(), packaged_model().body_links
    s, p = _groups(tree)[1]
    o = oracle_lib.PlenOracle(2)
    o.reset()
    emu = Emu(double=True)
    rec = np.stack([record_from_oracle_state(o.get_state(), e, dtype=np.float64) for e in range(2)])
    rec[:, 34] += 0.05                            # airborne: the difference is the free dynamics, not a contact decision
    st = oracle_state_from_record(rec)
    o.set_state(st)
    eq = oracle_lib.PlenOracle(2, tree=equivalent_tree(tree, links, s, p))
    eq.set_state(st)
    emu.set_mass(mass_rows(np.stack([s, s]), np.stack([p, p]), dtype=np.float64))
    try:
        emu.tick(rec, np.zeros((2, 18)), 1)
    finally:
        emu.set_mass(None)
    for e in range(2):
        o.tick(e)
        eq.tick(e)
    got = oracle_state_from_record(rec)["qvel"]
    assert np.abs(got - eq.get_state()["qvel"]).max() < 1e-7        # the model tables reach the device code as float32
    assert np.abs(got - o.get_state()["qvel"]).max() > 1e-4


def test_f32_unit_mass_rows_are_bit_identical_to_no_rows(oracle_lib):
    """Scale 1 and payload 0 in every row: the MASS instance reproduces the stock instance bit for bit (float32 build), through
    contact ticks, including M^-1 of the debug output."""
    n = 6
    o = oracle_lib.PlenOracle(n)
    o.reset()
    rng = np.random.default_rng(7)
    for _ in range(5):
        o.step(rng.uniform(-1, 1, (n, 18)))
    st = o.get_state()
    base = np.stack([record_from_oracle_state(st, e, dtype=np.float32) for e in range(n)])
    tg = rng.uniform(-1, 1, (n, 18)).astype(np.float32)
    emu = Emu(double=False)
    a, b = base.copy(), base.copy()
    ma = emu.tick(a, tg, 8, debug=True)
    emu.set_mass(mass_rows(np.ones((n, 19)), np.zeros((n, 4))))
    try:
        mb = emu.tick(b, tg, 8, debug=True)
    finally:
        emu.set_mass(None)
    assert a.tobytes() == b.tobytes()
    for x, y in zip(ma, mb):
        assert x.tobytes() == y.tobytes()
    assert np.abs(a - base).max() > 0                 # the robots moved


def test_f64_mass_rows_equal_an_equivalent_model():
    """The float64 build of the device source with mass rows against the same build run on a model whose lane tables hold the
    scaled bodies and the folded payload (payloads at arbitrary offsets): M^-1 and one free-flight tick agree to the float32
    rounding of the model tables (measured <= 7e-8 relative in M^-1, 1.6e-7 in the velocities)."""
    from mass_util import equivalent_model
    from parity_util import random_flight_state
    from plen_ml_walk_b200._abi import model_to_c
    rng = np.random.default_rng(6)
    groups = [(np.full(19, 1.25), np.zeros(4)), (rng.uniform(0.6, 1.5, 19), np.array([0.03, 0.01, -0.02, 0.03])),
              (np.ones(19), np.array([0.2, -0.03, 0.02, 0.05])), (rng.uniform(0.8, 1.2, 19), np.array([0.08, 0.0, 0.0, -0.01]))]
    qpos, qvel = random_flight_state(np.random.default_rng(1), 1)
    st = dict(qpos=qpos, qvel=qvel, lam_n=np.zeros((1, 8)), in_manifold=np.zeros((1, 8), dtype=np.int32),
              book_i=np.zeros((1, 5), dtype=np.int32), book_f=np.zeros((1, 16)))
    rec0 = record_from_oracle_state(st, 0, dtype=np.float64)[None]
    for s, p in groups:
        emu = Emu(double=True)
        emu.set_mass(mass_rows(s[None], p[None], dtype=np.float64))
        a = rec0.copy()
        try:
            m1 = emu.tick(a, np.zeros((1, 18)), 1, debug=True)[0]
        finally:
            emu.set_mass(None)
        eq = Emu(double=True)
        eq.model = model_to_c(equivalent_model(packaged_model(), s, p))
        b = rec0.copy()
        m2 = eq.tick(b, np.zeros((1, 18)), 1, debug=True)[0]
        assert np.abs((m1 - m2) / np.sqrt(np.outer(np.diag(m2), np.diag(m2)))).max() < 1e-6
        assert np.abs(a[:, :24] - b[:, :24]).max() < 1e-6
