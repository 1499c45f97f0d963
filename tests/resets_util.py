"""TEST-ONLY helpers for the per-robot reset states (plen_settle_env_resets): the start state of a pose (x, y, z, yaw) built
independently of the device code, the float64 oracle's settle from such poses, and the warp-emulation harness
(tests/emu/emu_resets.cpp) that exports the device's start_record."""
import ctypes as C
import os
import subprocess

import numpy as np

from emu_util import _DEPS, ROOT, Emu

EMU_RESETS_SRC = os.path.join(ROOT, "tests", "emu", "emu_resets.cpp")
EMU_RESETS_LIB = os.path.join(ROOT, "tests", "emu", "libplen_emu_resets.so")


def start_qpos(poses):
    """poses [n,4] (x, y, z, yaw) -> qpos [n,25] float32: base at (x, y, z), quaternion (0, 0, sin(yaw/2), cos(yaw/2)) from the
    float32 yaw, the half-angle functions in float64 rounded once (as start_record does), joints 0."""
    p = np.asarray(poses, dtype=np.float32).reshape(-1, 4)
    h = 0.5 * p[:, 3].astype(np.float64)
    q = np.zeros((p.shape[0], 25), np.float32)
    q[:, 0:3] = p[:, 0:3]
    q[:, 5] = np.sin(h).astype(np.float32)
    q[:, 6] = np.cos(h).astype(np.float32)
    return q


def oracle_settle(oracle_lib, poses, tree=None, setup=None, manifold_mode=0):
    """The reference's reset procedure (plen_env.py:558-574) in float64 from each pose: teleport (zero joints, velocities,
    targets and contact cache, empty manifolds), reset_ticks ticks, observe.  setup(cfg) may scale constants.
    -> (oracle, obs [n,26])"""
    poses = np.asarray(poses, dtype=np.float32).reshape(-1, 4)
    n = poses.shape[0]
    o = oracle_lib.PlenOracle(n, tree=tree)
    o.cfg.manifold_mode = int(manifold_mode)
    if setup is not None:
        setup(o.cfg)
    o.set_state({"qpos": start_qpos(poses).astype(np.float64)})        # every other field is 0 from plen_oracle_init_state
    obs = np.zeros((n, 26))
    for e in range(n):
        for _ in range(int(o.cfg.reset_ticks)):
            o.tick(e)
        obs[e] = o.observe(e)[0]
    return o, obs


def build_emu_resets(double=False):
    lib = EMU_RESETS_LIB.replace(".so", "_f64.so") if double else EMU_RESETS_LIB
    deps = _DEPS + [EMU_RESETS_SRC]
    if os.path.exists(lib) and all(os.path.getmtime(lib) >= os.path.getmtime(d) for d in deps):
        return lib
    subprocess.check_call(["g++", "-O1", "-std=c++20", "-pthread", "-fPIC", "-shared", "-ffp-contract=off",
                           "-I", ROOT, "-o", lib, EMU_RESETS_SRC] + (["-DPLEN_EMU_DOUBLE"] if double else []))
    return lib


class EmuResets(Emu):
    """Emu whose library also exports the device's start_record; settle() is the emulated plen_settle_env_resets."""

    def __init__(self, joint_act=False, double=False):
        super().__init__(joint_act=joint_act, double=double)
        self.L = C.CDLL(build_emu_resets(double))        # a superset of emu_warp.cpp's exports, same precision
        assert self.L.emu_real_bytes() == np.dtype(self.real).itemsize
        self.L.emu_default_config(C.byref(self.cfg), int(joint_act))

    def start_record(self, poses):
        poses = np.ascontiguousarray(np.asarray(poses, dtype=np.float32).reshape(-1, 4), dtype=self.real)
        rec = np.zeros((poses.shape[0], 96), dtype=self.real)
        for e in range(poses.shape[0]):
            self.L.emu_start_record(poses[e].ctypes.data_as(C.c_void_p), rec[e].ctypes.data_as(C.c_void_p))
        return rec

    def settle(self, poses):
        """start records, reset_ticks ticks with zero targets, observation -> (records [n,96], obs [n,26])"""
        rec = self.start_record(poses)
        self.tick(rec, np.zeros((rec.shape[0], 18)), int(self.cfg.reset_ticks))
        return rec, self.observe(rec)
