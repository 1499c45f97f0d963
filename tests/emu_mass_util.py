"""TEST-ONLY helpers for the MASS instance of the device code (per-robot mass rows, plen_set_env_mass) in the warp emulation:
build tests/emu/libplen_emu_mass.so (tests/emu/emu_mass.cpp on top of the emu_warp.cpp harness) and drive it like emu_util.Emu."""
import ctypes as C
import os
import subprocess

import numpy as np

from emu_util import _DEPS, ROOT, Emu

EMU_MASS_SRC = os.path.join(ROOT, "tests", "emu", "emu_mass.cpp")
EMU_MASS_LIB = os.path.join(ROOT, "tests", "emu", "libplen_emu_mass.so")


def build_emu_mass(double=False):
    lib = EMU_MASS_LIB.replace(".so", "_f64.so") if double else EMU_MASS_LIB
    deps = _DEPS + [EMU_MASS_SRC]
    if os.path.exists(lib) and all(os.path.getmtime(lib) >= os.path.getmtime(d) for d in deps):
        return lib
    subprocess.check_call(["g++", "-O1", "-std=c++20", "-pthread", "-fPIC", "-shared", "-ffp-contract=off",
                           "-I", ROOT, "-o", lib, EMU_MASS_SRC] + (["-DPLEN_EMU_DOUBLE"] if double else []))
    return lib


def mass_rows(scale, payload, dtype=np.float32):
    """[n,19] body mass scales and [n,4] torso payloads -> [n,32] mass rows in the layout plen_set_env_mass writes (word 0 and
    words 6..23: the scale of that lane's body, words 24..27: the payload, the rest 1)."""
    scale, payload = np.asarray(scale, dtype=np.float64), np.asarray(payload, dtype=np.float64)
    rows = np.ones((scale.shape[0], 32), dtype=dtype)
    rows[:, 0] = scale[:, 0]
    rows[:, 6:24] = scale[:, 1:]
    rows[:, 24:28] = payload
    return rows


class EmuMass(Emu):
    """Emu whose tick runs the MASS instance of the dynamics while mass rows are set (set_mass), the stock one otherwise."""

    def __init__(self, joint_act=False, double=False):
        super().__init__(joint_act=joint_act, double=double)
        self.M = C.CDLL(build_emu_mass(double))
        self._rows = None

    def set_mass(self, rows):
        """rows: [n,32] mass rows (mass_rows, dtype self.real); None switches back to the stock instance."""
        self._rows = None if rows is None else np.ascontiguousarray(rows, dtype=self.real)

    def tick(self, rec, targets, n_ticks=1, debug=False):
        if self._rows is None:
            return super().tick(rec, targets, n_ticks, debug)
        n = rec.shape[0]
        assert self._rows.shape == (n, 32)
        targets = np.ascontiguousarray(targets, dtype=self.real).reshape(n, 18)
        minv = np.zeros((24, 24), dtype=self.real)
        pos = np.zeros((24, 3), dtype=self.real)
        rot = np.zeros((24, 3, 3), dtype=self.real)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self.M.emu_tick_mass(C.byref(self.model), C.byref(self.cfg), vp(rec), vp(targets), vp(self._rows), n, n_ticks,
                             vp(minv) if debug else None, vp(pos) if debug else None, vp(rot) if debug else None)
        iters = rec[:, 79].astype(np.int32)
        return (minv, pos, rot, iters) if debug else iters
