"""TEST-ONLY helpers: build and drive tests/cuda/libtick_harness.so, the library (plen_b200.cu) with the two halves of a
physics tick exported one by one (th_dyn, th_rank, th_solve), so GPU tests can read and write the solve records, extension
records, sort keys and permutation that k_dyn, k_rank and k_solve pass to each other."""
import ctypes as C
import os
import subprocess

import numpy as np

from plen_ml_walk_b200.build import NVCC_FLAGS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS_SRC = os.path.join(ROOT, "tests", "cuda", "tick_harness.cu")
HARNESS_LIB = os.path.join(ROOT, "tests", "cuda", "libtick_harness.so")
_CSRC = os.path.join(ROOT, "plen_ml_walk_b200", "csrc")
_DEPS = [HARNESS_SRC] + [os.path.join(_CSRC, f) for f in ("plen_b200.cu", "plen_device.cuh", "plen_solve.cuh", "plen_env.cuh",
                                                          "plen_host_tables.h")] + \
        [os.path.join(ROOT, "include", "plen_b200.h")]

SR_WORDS, XR_WORDS, MAN_WORDS, MR_WORDS = 1600, 976, 52, 32


def nvcc():
    return os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def build_harness():
    if os.path.exists(HARNESS_LIB) and all(os.path.getmtime(HARNESS_LIB) >= os.path.getmtime(d) for d in _DEPS):
        return HARNESS_LIB
    p = subprocess.run([nvcc()] + NVCC_FLAGS + ["-ccbin", "/usr/bin/g++", "-I", ROOT, "-o", HARNESS_LIB, HARNESS_SRC],
                       capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError("nvcc failed building the tick harness:\n" + p.stdout + p.stderr)
    return HARNESS_LIB


_lib = None


def load_harness():
    global _lib
    if _lib is None:
        from plen_ml_walk_b200._abi import PlenConfigC, PlenModelC
        L = C.CDLL(build_harness())
        vp, ip = C.c_void_p, C.c_int
        L.plen_default_config.argtypes = [C.POINTER(PlenConfigC), ip]
        L.plen_create.argtypes = [C.POINTER(PlenConfigC), C.POINTER(PlenModelC), ip, ip]
        L.plen_create.restype = vp
        L.plen_destroy.argtypes = [vp]
        L.plen_destroy.restype = None
        L.plen_last_error.argtypes = [vp]
        L.plen_last_error.restype = C.c_char_p
        L.plen_tick.argtypes = [vp, vp, ip, vp]
        L.plen_set_env_mass.argtypes = [vp] * 4
        L.th_buffers.argtypes = [vp, C.POINTER(C.c_void_p)]
        L.th_dyn.argtypes = [vp, vp, vp]
        L.th_rank.argtypes = [vp, vp]
        L.th_solve.argtypes = [vp, ip, vp]
        L.th_set_solver.argtypes = [vp, ip, C.c_float, ip]
        L.th_set_solver.restype = None
        _lib = L
    return _lib


class _Dev:
    """__cuda_array_interface__ view of raw device memory, for torch.as_tensor"""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = dict(shape=tuple(shape), typestr=typestr, data=(int(ptr), False), version=3, strides=None)


class TickCtx:
    """One context of the harness library (its own plen_create) with torch views of its per-robot buffers:
    state [n,96], srec [n,SR_WORDS], srx [n,XR_WORDS], key [n] uint8, perm [tiles*1024] int32, xgroups [tiles] int32,
    man [n,52], scale [n,4], mass [n,32] (None where the context holds no such buffer)."""

    def __init__(self, n, overrides=None):
        import torch
        from plen_ml_walk_b200._abi import PlenConfigC, model_to_c
        from plen_ml_walk_b200.urdf_loader import packaged_model
        self.L = load_harness()
        self.n = int(n)
        self.cfg = PlenConfigC()
        self.L.plen_default_config(C.byref(self.cfg), 0)
        self.cfg.auto_reset = 0
        for k, v in (overrides or {}).items():
            setattr(self.cfg, k, v)
        self._model = model_to_c(packaged_model())
        self.ctx = self.L.plen_create(C.byref(self.cfg), C.byref(self._model), self.n, torch.cuda.current_device())
        if not self.ctx:
            raise RuntimeError("plen_create failed: %s" % self.L.plen_last_error(None).decode())
        self.tiles = (self.n + 1023) // 1024
        self._views()

    def _views(self):
        import torch
        p = (C.c_void_p * 9)()
        assert self.L.th_buffers(self.ctx, p) == self.n
        n, t = self.n, self.tiles

        def v(ptr, shape, ty):
            return None if not ptr else torch.as_tensor(_Dev(ptr, shape, ty), device="cuda")
        self.state = v(p[0], (n, 96), "<f4")
        self.srec = v(p[1], (n, SR_WORDS), "<f4")
        self.srx = v(p[2], (n, XR_WORDS), "<f4")
        self.key = v(p[3], (n,), "|u1")
        self.perm = v(p[4], (t * 1024,), "<i4")
        self.xgroups = v(p[5], (t,), "<i4")
        self.man = v(p[6], (n, MAN_WORDS), "<f4")
        self.scale = v(p[7], (n, 4), "<f4")
        self.mass = v(p[8], (n, MR_WORDS), "<f4")

    def _st(self):
        import torch
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def _ck(self, rc, what):
        if rc != 0:
            raise RuntimeError("%s: error %d" % (what, rc))

    def set_mass(self, mass_scale, payload):
        """plen_set_env_mass with [n,19] / [n,4] arrays; allocates the mass rows (self.mass)"""
        import torch
        a = torch.as_tensor(np.ascontiguousarray(mass_scale, np.float32), device="cuda")
        b = torch.as_tensor(np.ascontiguousarray(payload, np.float32), device="cuda")
        self._ck(self.L.plen_set_env_mass(self.ctx, a.data_ptr(), b.data_ptr(), self._st()), "plen_set_env_mass")
        torch.cuda.synchronize()
        self._views()

    def dyn(self, targets=None):
        self._ck(self.L.th_dyn(self.ctx, None if targets is None else targets.data_ptr(), self._st()), "th_dyn")

    def rank(self):
        self._ck(self.L.th_rank(self.ctx, self._st()), "th_rank")

    def solve(self, merged):
        self._ck(self.L.th_solve(self.ctx, int(merged), self._st()), "th_solve")

    def tick(self, targets=None, n_ticks=1):
        self._ck(self.L.plen_tick(self.ctx, None if targets is None else targets.data_ptr(), n_ticks, self._st()), "plen_tick")

    def set_solver(self, iterations=50, residual_threshold=1e-7, merge_max=32768):
        """PGS iteration cap / early-exit threshold of the later solves, and the largest batch plen_tick solves merged"""
        self.L.th_set_solver(self.ctx, int(iterations), float(residual_threshold), int(merge_max))

    def close(self):
        if self.ctx:
            self.L.plen_destroy(self.ctx)
            self.ctx = None
