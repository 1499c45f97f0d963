"""TEST-ONLY helpers: build and drive tests/cuda/libtd3_gemm_harness.so, the TD3 learner's GEMM dispatch (launch() of
plen_td3_learn.cu with its five kernels) exported on its own so tests can check every product kind against float64."""
import ctypes as C
import os
import subprocess

from plen_ml_walk_b200.build import NVCC_FLAGS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS_SRC = os.path.join(ROOT, "tests", "cuda", "td3_gemm_harness.cu")
HARNESS_LIB = os.path.join(ROOT, "tests", "cuda", "libtd3_gemm_harness.so")
_CSRC = os.path.join(ROOT, "plen_ml_walk_b200", "csrc")
_DEPS = [HARNESS_SRC] + [os.path.join(_CSRC, f) for f in ("plen_td3.cu", "plen_td3_learn.cu", "plen_gemm_tc.cuh",
                                                          "plen_tc_common.cuh")] + \
        [os.path.join(ROOT, "include", "plen_b200.h")]

# epilogue ids of plen_td3_learn.cu
EPI_NONE, EPI_BIAS, EPI_BIAS_RELU, EPI_BIAS_TANH, EPI_BIAS_TANH_NOISE, EPI_RELUMASK, EPI_TANHGRAD = range(7)


def nvcc():
    return os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def build_harness():
    if os.path.exists(HARNESS_LIB) and all(os.path.getmtime(HARNESS_LIB) >= os.path.getmtime(d) for d in _DEPS):
        return HARNESS_LIB
    p = subprocess.run([nvcc()] + NVCC_FLAGS + ["-ccbin", "/usr/bin/g++", "-I", ROOT, "-o", HARNESS_LIB, HARNESS_SRC],
                       capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError("nvcc failed building the TD3 GEMM harness:\n" + p.stdout + p.stderr)
    return HARNESS_LIB


_lib = None


def load_harness():
    global _lib
    if _lib is None:
        L = C.CDLL(build_harness())
        L.harness_gemm.argtypes = [C.POINTER(C.c_void_p), C.POINTER(C.c_longlong), C.POINTER(C.c_int), C.POINTER(C.c_float),
                                   C.c_ulonglong, C.c_void_p]
        L.harness_gemm.restype = C.c_int
        L.harness_tc_timed_out.restype = C.c_int
        _lib = L
    return _lib


def gemm(a, b, c, *, M, N, K, az=0, am, ak, bz=0, bk, bn, cz=0, ldc, nz=1, epi=EPI_NONE, bias=None, bias_z=0,
         aux=None, aux_z=0, ld_aux=0, p=(0.0, 0.0, 0.0), seed=0, rowsum=None, rowsum_z=0, tc=False):
    """One launch() on the current stream.  a, b, c, bias, aux, rowsum: CUDA float32 tensors or raw device addresses (int)
    of their first element; the strides are in elements, as in plen_td3_learn.cu's Gemm."""
    import torch
    L = load_harness()
    addr = lambda t: 0 if t is None else (t if isinstance(t, int) else t.data_ptr())
    ptr = (C.c_void_p * 6)(*[addr(t) or None for t in (a, b, c, bias, aux, rowsum)])
    st = (C.c_longlong * 12)(az, am, ak, bz, bk, bn, cz, ldc, bias_z, aux_z, ld_aux, rowsum_z)
    dim = (C.c_int * 6)(M, N, K, nz, epi, 1 if tc else 0)
    pf = (C.c_float * 3)(*p)
    rc = L.harness_gemm(ptr, st, dim, pf, seed & (2 ** 64 - 1), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    if rc != 0:
        raise RuntimeError("harness_gemm: cudaError %d" % rc)
