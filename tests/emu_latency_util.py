"""TEST-ONLY helpers for env steps with per-robot command latency (plen_set_env_latency) in the warp emulation: build
tests/emu/libplen_emu_latency.so (tests/emu/emu_latency.cpp on top of the emu_warp.cpp harness) and drive it like emu_util.Emu."""
import ctypes as C
import os
import subprocess

import numpy as np

from emu_util import _DEPS, ROOT, Emu

EMU_LATENCY_SRC = os.path.join(ROOT, "tests", "emu", "emu_latency.cpp")
EMU_LATENCY_LIB = os.path.join(ROOT, "tests", "emu", "libplen_emu_latency.so")
LAT_WORDS = 96      # LAT_SLOTS (3) ring rows of 32 words per robot (plen_device.cuh)


def build_emu_latency():
    deps = _DEPS + [EMU_LATENCY_SRC]
    lib = EMU_LATENCY_LIB
    if os.path.exists(lib) and all(os.path.getmtime(lib) >= os.path.getmtime(d) for d in deps):
        return lib
    subprocess.check_call(["g++", "-O1", "-std=c++20", "-pthread", "-fPIC", "-shared", "-ffp-contract=off",
                           "-I", ROOT, "-o", lib, EMU_LATENCY_SRC])
    return lib


class EmuLatency(Emu):
    """float32 Emu with env steps that run the latency prologue of k_dyn (step_latency) and env_post alone (post)."""

    def __init__(self, joint_act=False):
        super().__init__(joint_act=joint_act)
        self.X = C.CDLL(build_emu_latency())

    def latency_source(self, d, k, S, ep_t):
        return int(self.X.emu_latency_source(int(d), int(k), int(S), int(ep_t)))

    def latency_slot(self, ep_t, s):
        return int(self.X.emu_latency_slot(int(ep_t), int(s)))

    def new_ring(self, last):
        """[n,96] history ring seeded the way the first plen_set_env_latency call does: every row holds `last` [n,18]."""
        ring = np.zeros((last.shape[0], LAT_WORDS), dtype=np.float32)
        for s in range(3):
            ring[:, 32 * s + 6:32 * s + 24] = last
        return ring

    @staticmethod
    def _outputs(n):
        return (np.zeros((n, 26), np.float32), np.zeros(n, np.float32), np.zeros(n, np.uint8), np.zeros(n, np.uint8),
                np.zeros((n, 26), np.float32))

    def step_latency(self, rec, actions, ring, ticks, snapshot):
        """One env step with command latency; rec [n,96] and ring [n,96] are updated in place.  -> (obs, reward, done,
        raw targets [n,18] of this step)"""
        n = rec.shape[0]
        actions = np.ascontiguousarray(actions, dtype=np.float32).reshape(n, 18)
        ticks = np.ascontiguousarray(ticks, dtype=np.int32).reshape(n)
        tgt = np.zeros((n, 18), np.float32)
        obs, rew, done, tmo, tobs = self._outputs(n)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self.X.emu_step_latency(C.byref(self.model), C.byref(self.cfg), vp(rec), vp(actions), vp(tgt), vp(ring), vp(ticks), n,
                                vp(obs), vp(rew), vp(done), vp(tmo), vp(tobs), vp(snapshot))
        return obs, rew, done.astype(bool), tgt

    def post(self, rec, snapshot):
        """env_post of every robot (rec updated in place) -> (obs, reward, done)"""
        n = rec.shape[0]
        obs, rew, done, tmo, tobs = self._outputs(n)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self.X.emu_post(C.byref(self.model), C.byref(self.cfg), vp(rec), n, vp(obs), vp(rew), vp(done), vp(tmo), vp(tobs),
                        vp(snapshot))
        return obs, rew, done.astype(bool)
