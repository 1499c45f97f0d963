"""Build libplen_b200.so in-tree with nvcc for sm_100a (the only target; there is no CPU build)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRCS = [os.path.join(HERE, "csrc", "plen_b200.cu"), os.path.join(HERE, "csrc", "plen_td3.cu"),
        os.path.join(HERE, "csrc", "plen_td3_learn.cu"), os.path.join(HERE, "csrc", "plen_actor_tc.cu")]
DEPS = SRCS + [os.path.join(HERE, "csrc", f) for f in ("plen_device.cuh", "plen_solve.cuh", "plen_env.cuh", "plen_host_tables.h", "plen_tc_common.cuh", "plen_gemm_tc.cuh")] + \
       [os.path.join(ROOT, "include", "plen_b200.h")]
OUT = os.path.join(HERE, "libplen_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--shared",
    "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-cudart", "static",
]


def build(force: bool = False, verbose: bool = False) -> str:
    if (not force) and os.path.exists(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(d) for d in DEPS):
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-ccbin", "/usr/bin/g++", "-I", ROOT, "-o", OUT] + SRCS
    p = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or p.returncode != 0:
        sys.stderr.write(p.stdout + p.stderr)
    if p.returncode != 0:
        raise RuntimeError("nvcc failed building libplen_b200.so")
    with open(os.path.join(HERE, "csrc", "ptxas_info.txt"), "w") as f:
        # register / spill report of every kernel; compile times would only be noise.  Not tracked by git: the kernel names
        # of anonymous namespaces carry a hash of the build directory, so every checkout writes a different file
        f.write("".join(l for l in p.stderr.splitlines(True) if "Compile time" not in l))
    return OUT


if __name__ == "__main__":
    print(build(force=True, verbose=True))
