"""Builds chronoclust_b200/libchronoclust_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python chronoclust_b200/build.py [--force] [--debug]

--debug builds libchronoclust_b200_debug.so instead: the same sources with -DCCB_DEBUG, which adds the diagnostics of
csrc/debug.h (per-key cycle counters of the replay kernel, event counters, the round-by-round trace ring).  The
product library never contains them.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "api.cu")
DEPS = [os.path.join(HERE, "csrc", f) for f in ("api.cu", "common.cuh", "nearest.cuh", "online.cuh", "offline.cuh",
                                                "engine.cuh", "stats.cuh", "debug.h", "asinh.h")]
DEPS.append(os.path.join(os.path.dirname(HERE), "include", "chronoclust_b200.h"))
SO = os.path.join(HERE, "libchronoclust_b200.so")
SO_DEBUG = os.path.join(HERE, "libchronoclust_b200_debug.so")
HOSTIO_SRC = os.path.join(HERE, "csrc", "hostio.c")
HOSTIO_DEPS = [HOSTIO_SRC, os.path.join(HERE, "csrc", "asinh.h")]
HOSTIO_SO = os.path.join(HERE, "libccb_hostio.so")

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-fmad=false",            # parity: the reference never contracts mul+add (SURVEY Appendix C)
    "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-shared", "-Xptxas", "-v" if os.environ.get("CCB_PTXAS_V") else "-O3",
    # the kernels of this one translation unit are optimised in 8 groups -- a FIXED count, so that the binary does not
    # depend on how many cores the build host has (`--split-compile 0` made it irreproducible)
    "--split-compile", "8",
]


def nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def build(force=False, verbose=False, debug=False):
    so = SO_DEBUG if debug else SO
    if not force and os.path.exists(so) and all(os.path.getmtime(so) >= os.path.getmtime(d) for d in DEPS):
        return so
    cmd = [nvcc()] + NVCC_FLAGS + (["-DCCB_DEBUG"] if debug else []) + ["-o", so, SRC]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return so


def build_hostio(force=False, verbose=False):
    """The host-side CSV writer and arcsinh transform (plain C, pthreads; no CUDA): chronoclust_b200/libccb_hostio.so.
    -ffp-contract=off: csrc/asinh.h gives the device's bits only when no a * b + c is fused (GNU C's default is fast)."""
    if not force and os.path.exists(HOSTIO_SO) and all(os.path.getmtime(HOSTIO_SO) >= os.path.getmtime(d)
                                                       for d in HOSTIO_DEPS):
        return HOSTIO_SO
    cmd = ["gcc", "-O2", "-std=gnu11", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-o", HOSTIO_SO, HOSTIO_SRC,
           "-lm"]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return HOSTIO_SO


if __name__ == "__main__":
    print(build_hostio(force="--force" in sys.argv, verbose=True))
    print(build(force="--force" in sys.argv, verbose=True, debug="--debug" in sys.argv))
