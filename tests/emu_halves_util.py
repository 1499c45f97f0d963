"""TEST-ONLY helpers for the two halves of a physics tick in the warp emulation: build tests/emu/libplen_emu_halves.so
(tests/emu/emu_halves.cpp on top of the emu_warp.cpp harness) and drive emu_dyn / emu_solve like emu_util.Emu; the record
layouts (plen_device.cuh SR_* / XR_*) and the state families the CPU and GPU tests of the halves share."""
import ctypes as C
import os
import subprocess

import numpy as np

from emu_util import _DEPS, ROOT, Emu, record_from_oracle_state

EMU_HALVES_SRC = os.path.join(ROOT, "tests", "emu", "emu_halves.cpp")
EMU_HALVES_LIB = os.path.join(ROOT, "tests", "emu", "libplen_emu_halves.so")

SR_WORDS, XR_WORDS = 1600, 16 + 3 * 4 * 80
KEY_EXT, MAX_BOX_POINTS = 125, 4
SR_PT, SR_BASE = 1536, 1576
SR_MAN = SR_BASE + 13            # manifold bits: an integer held in a float
XR_NX, XR_ROWS, XR_ROW_WORDS = 0, 16, 80
# solve-record blocks (plen_device.cuh): name -> (first word, end)
SR_BLOCKS = dict(G=(0, 960), B=(960, 1152), MRHS=(1152, 1184), MD=(1184, 1216), LDIR=(1216, 1248), LRHS=(1248, 1280),
                 VSTAR=(1280, 1312), Q=(1312, 1344), CRHS=(1344, 1408), CDINV=(1408, 1472), CD=(1472, 1536), PT=(1536, 1568),
                 LAMC=(1568, 1576), BASE=(1576, 1600))
# per-robot bound on |float32 - float64| of the velocities and cached impulses after k capped PGS sweeps without early exit
# on the same record, k = 1, 2, 4, 8 (a few times the worst cases measured: host float32 build 1.6e-4 / 7.8e-5 / 2.9e-4 /
# 1.4e-3, sm_100a build 7.7e-5 / 3.3e-4 / 5.2e-4 / 7.7e-4 on a B200; each sweep re-decides the clamps of the lateral pairs)
SWEEP_BOUND = {1: 8e-4, 2: 1.5e-3, 4: 2.5e-3, 8: 7e-3}


def build_emu_halves(double=False):
    lib = EMU_HALVES_LIB.replace(".so", "_f64.so") if double else EMU_HALVES_LIB
    deps = _DEPS + [EMU_HALVES_SRC]
    if os.path.exists(lib) and all(os.path.getmtime(lib) >= os.path.getmtime(d) for d in deps):
        return lib
    subprocess.check_call(["g++", "-O1", "-std=c++20", "-pthread", "-fPIC", "-shared", "-ffp-contract=off",
                           "-I", ROOT, "-o", lib, EMU_HALVES_SRC] + (["-DPLEN_EMU_DOUBLE"] if double else []))
    return lib


def _vp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class EmuHalves(Emu):
    """Emu with the two halves of a tick as separate calls (dyn, solve); every real array is self.real."""

    def __init__(self, joint_act=False, double=False):
        super().__init__(joint_act=joint_act, double=double)
        self.H = C.CDLL(build_emu_halves(double))
        assert self.H.emu_sr_words() == SR_WORDS and self.H.emu_xr_words() == XR_WORDS

    def _real(self, a, shape=None):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=self.real)
        return a if shape is None else a.reshape(shape)

    def dyn(self, rec, targets, scales=None, mass_rows=None, man=None, fill=0.0):
        """-> (solve records [n,SR_WORDS], extension records [n,XR_WORDS], keys [n] uint8).  rec is not changed; man ([n,52],
        self.real) is updated in place when given, as k_dyn updates the manifolds.  The words k_dyn does not write keep
        `fill`."""
        n = rec.shape[0]
        rec = self._real(rec)
        srec = np.full((n, SR_WORDS), fill, self.real)
        srx = np.full((n, XR_WORDS), fill, self.real)
        keys = np.zeros(n, np.uint8)
        if man is not None:
            assert man.dtype == self.real and man.flags.c_contiguous
        self.H.emu_dyn(C.byref(self.model), C.byref(self.cfg), _vp(rec), _vp(self._real(targets, (n, 18))),
                       _vp(self._real(scales, (n, 4))), _vp(self._real(mass_rows, (n, 32))), _vp(man), n, _vp(srec), _vp(srx),
                       _vp(keys))
        return srec, srx, keys

    def solve(self, rec, srec, srx, keys, order=None):
        """PGS + integration of the records in place (rec: [n,96] self.real); order: robots in solver-group order (entries >= n
        are invalid lanes), None = 0 .. n-1."""
        n = rec.shape[0]
        assert rec.dtype == self.real and rec.flags.c_contiguous
        srec, srx = self._real(srec), self._real(srx)
        keys = np.ascontiguousarray(keys, dtype=np.uint8)
        order = None if order is None else np.ascontiguousarray(order, dtype=np.int32)
        self.H.emu_solve(C.byref(self.model), C.byref(self.cfg), _vp(rec), _vp(srec), _vp(srx), _vp(keys), _vp(order),
                         0 if order is None else len(order), n)

    def set_solver(self, iterations, residual_threshold):
        self.cfg.solver_iterations = int(iterations)
        self.cfg.residual_threshold = float(residual_threshold)


def sort_keys(srec, srx):
    """k_dyn's sort key recomputed from the manifold bits and the box point count (plen_device.cuh)"""
    man = srec[:, SR_MAN].astype(np.int64)
    n0 = np.array([bin(m & 15).count("1") for m in man])
    n1 = np.array([bin((m >> 4) & 15).count("1") for m in man])
    nx = srx[:, XR_NX].astype(np.int64)
    return np.where(nx > 0, KEY_EXT + nx - 1, np.maximum(n0, n1) * 25 + n0 * 5 + n1).astype(np.uint8)


def real_noise(srec, srx, rng, rel):
    """srec / srx with every real-valued word scaled by (1 + rel * N(0, 1)); the integer-coded words (the manifold bits and the
    box point count) are kept, since flipping one of their bits changes the row set, not a value"""
    a = srec * (1.0 + rel * rng.standard_normal(srec.shape))
    a[:, SR_MAN] = srec[:, SR_MAN]
    b = srx * (1.0 + rel * rng.standard_normal(srx.shape))
    b[:, XR_NX] = srx[:, XR_NX]
    return a, b


# ---- state families: float32 state records [n,96] and raw servo targets [n,18] from oracle states
FAMILIES = ("contact", "fallen", "limits", "vclamp", "mass", "manifold")


def _euler_quat(ang):
    cr, sr, cp, sp, cy, sy = (f(ang[:, i] / 2) for i in range(3) for f in (np.cos, np.sin))
    return np.stack([sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy, cr * cp * sy - sr * sp * cy, cr * cp * cy + sr * sp * sy], 1)


def make_family(oracle_lib, fam, n, seed):
    """-> dict(rec [n,96] float32, tgt [n,18] float32, cfg (plen_config overrides), scales [n,4] | None,
    mass_scale [n,19] | None, payload [n,4] | None, man [n,52] float32 | None)"""
    rng = np.random.default_rng(seed)
    out = dict(cfg={}, scales=None, mass_scale=None, payload=None, man=None)
    o = oracle_lib.PlenOracle(n, n_threads=8)
    if fam == "manifold":
        o.cfg.manifold_mode = 1
        out["cfg"]["sole_manifold"] = 1
    if fam in ("contact", "vclamp", "mass", "manifold"):
        # teacher-forced contact states: oracle rollouts under random actions from the reset pose, each robot stopped after
        # its own number of steps (2..24), fallen robots restarted
        o.reset()
        st0 = o.get_state()
        stop = rng.integers(2, 25, n)
        snap = None
        for t in range(int(stop.max())):
            amp = 0.3 if fam == "manifold" else 1.0
            _, _, done, _ = o.step(rng.uniform(-amp, amp, (n, 18)))
            st = o.get_state()
            man = o.get_manifold() if fam == "manifold" else None
            if snap is None:
                snap = {k: v.copy() for k, v in st.items()}
                mans = man.copy() if man is not None else None
            sel = stop == t + 1
            for k in snap:
                snap[k][sel] = st[k][sel]
            if man is not None:
                mans[sel] = man[sel]
            for e in np.where(done)[0]:
                o.reset_one(int(e))
        st = snap
        if fam == "contact":
            # every eighth robot: the settled reset pose pressed 1-3 mm into the ground, all four corners of both soles in
            # contact (8-point robots, which random rollouts rarely reach)
            sel = np.arange(n) % 8 == 0
            for k in st:
                st[k][sel] = st0[k][sel]
            st["qpos"][sel, 2] -= rng.uniform(0.001, 0.003, int(sel.sum()))
        if fam == "manifold":
            out["man"] = mans.astype(np.float32)
    else:
        st = o.get_state()
        if fam == "fallen":
            # robots lying on the ground, one box vertex 2 mm under it (test_box_contacts_on_fallen_poses)
            o.reset()
            st = o.get_state()
            st["qpos"][:, 7:] = rng.uniform(-0.7, 0.7, (n, 18))
            ang = rng.uniform(-0.3, 0.3, (n, 3))
            ang[:, 2] = rng.uniform(-3, 3, n)
            ang[np.arange(n), rng.integers(0, 2, n)] = rng.choice([-1, 1], n) * rng.uniform(1.2, 1.9, n)
            st["qpos"][:, 3:7] = _euler_quat(ang)
            st["qpos"][:, 2] = 0.5
            st["qvel"][:, :6] = rng.normal(size=(n, 6)) * 0.1
            st["qvel"][:, 6:] = rng.normal(size=(n, 18)) * 0.5
            st["lam_n"][:] = 0
            st["in_manifold"][:] = 0
            o.set_state(st)
            for e in range(n):
                pos, rot = o.fk(e)
                low = min((pos[b["link"] + 1] + rot[b["link"] + 1] @ np.array(b["center"]))[2] -
                          np.abs((rot[b["link"] + 1] @ np.array(b["rot"]))[2]) @ np.array(b["half"]) for b in o.tree["boxes"])
                lowf = min((pos[f["link"] + 1] + np.array(f["points"]) @ rot[f["link"] + 1].T)[:, 2].min() - 0.001 for f in o.tree["feet"])
                st["qpos"][e, 2] -= max(low, lowf - 0.004) + 0.002
        elif fam == "limits":
            # airborne robots with joints beyond the +-1.7 rad URDF limits in some lanes only; every fourth robot has none
            from parity_util import random_flight_state
            st["qpos"], st["qvel"] = random_flight_state(rng, n)
            st["qvel"][:, 6:] *= 0.25
            viol = rng.random((n, 18)) < 0.1
            viol[::4] = False
            sign = np.where(rng.random((n, 18)) < 0.5, -1.0, 1.0)
            st["qpos"][:, 7:] = np.where(viol, sign * (1.7 + rng.uniform(0.002, 0.2, (n, 18))), st["qpos"][:, 7:])
            st["lam_n"][:] = 0
            st["in_manifold"][:] = 0
        o.set_state(st)
        st = o.get_state()
    if fam == "vclamp":
        # some joint and base velocities at (or past) max_coord_velocity = 100: v* is clamped there
        hit = rng.random((n, 24)) < 0.15
        st["qvel"] = np.where(hit, np.where(rng.random((n, 24)) < 0.5, -1.0, 1.0) * rng.uniform(99.0, 104.0, (n, 24)), st["qvel"])
    if fam == "mass":
        out["scales"] = np.stack([rng.uniform(0.5, 1.5, n), rng.uniform(0.6, 1.4, n), rng.uniform(0.6, 1.4, n), np.ones(n)], 1).astype(np.float32)
        out["mass_scale"] = rng.uniform(0.7, 1.4, (n, 19)).astype(np.float32)
        pay = np.zeros((n, 4), np.float32)
        pay[:, 0] = rng.uniform(0.0, 0.15, n)
        pay[:, 1:] = rng.uniform(-0.03, 0.03, (n, 3))
        out["payload"] = pay
    out["rec"] = np.stack([record_from_oracle_state(st, e, dtype=np.float32) for e in range(n)])
    out["tgt"] = rng.uniform(-1.0, 1.0, (n, 18)).astype(np.float32)
    out["state"] = st
    return out


def record_errors(a, b):
    """Per-robot worst element error of solve records a against the reference b, each element relative to its row's block
    maximum of |b|: a 32-word row of G or B (one column of G / one base row), the whole block elsewhere.  -> {block: [n]}"""
    out = {}
    for name, (lo, hi) in SR_BLOCKS.items():
        w = 32 if name in ("G", "B") else hi - lo
        d = np.abs(a[:, lo:hi] - b[:, lo:hi]).reshape(a.shape[0], -1, w)
        sc = np.abs(b[:, lo:hi]).reshape(a.shape[0], -1, w).max(2, keepdims=True)
        out[name] = np.where(sc > 0, d / np.where(sc > 0, sc, 1.0), d).max((1, 2))
    return out


# parts of a box-contact row of the extension record: Jx, Bx, Bb (base delta-v) and the row scalars (rhs, 1/d, d)
XR_PARTS = dict(Jx=(0, 32), Bx=(32, 64), Bb=(64, 70), scalars=(70, 73))


def ext_errors(a, b):
    """Per-robot worst element error of the extension records a against b, part by part, relative to the part's maximum
    over the robot's rows.  -> {part: [n]}"""
    n = a.shape[0]
    ra = a[:, XR_ROWS:].reshape(n, 3 * MAX_BOX_POINTS, XR_ROW_WORDS)
    rb = b[:, XR_ROWS:].reshape(n, 3 * MAX_BOX_POINTS, XR_ROW_WORDS)
    out = {}
    for name, (lo, hi) in XR_PARTS.items():
        d = np.abs(ra[:, :, lo:hi] - rb[:, :, lo:hi]).max((1, 2))
        sc = np.abs(rb[:, :, lo:hi]).max((1, 2))
        out[name] = np.where(sc > 0, d / np.where(sc > 0, sc, 1.0), d)
    return out


def structure(srec, srx, keys):
    """The discrete decisions of k_dyn per robot as one int64 row: key, manifold bits, box point count, the joints with a
    limit row (bit mask of the nonzero limit directions) and the occupied contact slots of SR_PT."""
    ld = (srec[:, 1216:1248] != 0) @ (1 << np.arange(32, dtype=np.int64))
    pt = (srec[:, SR_PT:SR_PT + 32].reshape(-1, 8, 4) != 0).any(2) @ (1 << np.arange(8, dtype=np.int64))
    return np.stack([keys.astype(np.int64), srec[:, SR_MAN].astype(np.int64), srx[:, XR_NX].astype(np.int64), ld, pt], 1)
