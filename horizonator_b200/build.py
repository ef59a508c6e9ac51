"""Builds the native pieces of horizonator_b200 in-tree (no JIT cache): 

  horizonator_b200/lib/libhorizonator.so   the product: C ABI of include/*.h, CUDA kernels for sm_100a
  horizonator_b200/lib/libsynth.so         synthetic SRTM tile generator (tests/bench input data)
  horizonator_b200/bin/horizonator-standalone   GL-free command-line renderer (cli/, plain C on the C ABI)

nvcc cross-compiles for sm_100a without a GPU.  -fmad=false: see csrc/hz_math.cuh.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "lib")

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-fmad=false",
    "-Xcompiler", "-fPIC,-O2,-ffp-contract=off,-Wall",
    "-shared",
    "-Xlinker", "-soname=libhorizonator.so.0",   # ABI 0, as the reference's Makefile:5-6
]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA renderer cannot be built (there is no CPU fallback)")


def build_library(force=False, extra_flags=(), verbose=False, name="libhorizonator.so"):
    """name: another file name for a compile-time variant (extra_flags), loaded with HORIZONATOR_LIBRARY=<path>."""
    os.makedirs(LIB, exist_ok=True)
    out = os.path.join(LIB, name)
    srcs = [os.path.join(CSRC, f) for f in ("hz_kernels.cu", "hz_api.cpp", "hz_dem.cpp")]
    deps = srcs + [os.path.join(CSRC, f) for f in ("hz_device.h", "hz_math.cuh", "hz_project.h")] + \
        [os.path.join(ROOT, "include", f) for f in ("horizonator.h", "horizonator-batch.h", "dem.h", "util.h")] + \
        [os.path.abspath(__file__)]
    if force or _newer(out, deps):
        cmd = [find_nvcc()] + NVCC_FLAGS + list(extra_flags) + ["-I", os.path.join(ROOT, "include"), "-I", CSRC, "-o", out] + srcs
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
    if name != "libhorizonator.so":
        return out
    # the SONAME is libhorizonator.so.0: give the dynamic loader that name too
    link = out + ".0"
    if not os.path.islink(link) and not os.path.exists(link):
        os.symlink(os.path.basename(out), link)
    return out


def build_synth(force=False):
    os.makedirs(LIB, exist_ok=True)
    out = os.path.join(LIB, "libsynth.so")
    src = os.path.join(ROOT, "tools", "synth_hgt.c")
    if force or _newer(out, [src]):
        subprocess.run(["/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc",
                        "-O2", "-fopenmp", "-shared", "-fPIC", src, "-o", out, "-lm"], check=True)
    return out


def build_cli(force=False):
    """cli/horizonator-standalone.c -> horizonator_b200/bin/horizonator-standalone (plain C against the C ABI)."""
    bindir = os.path.join(HERE, "bin")
    os.makedirs(bindir, exist_ok=True)
    out = os.path.join(bindir, "horizonator-standalone")
    src = os.path.join(ROOT, "cli", "horizonator-standalone.c")
    lib = os.path.join(LIB, "libhorizonator.so")
    if force or _newer(out, [src, lib]):
        subprocess.run(["/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc", "-O2", "-std=gnu99", "-Wall",
                        "-I", os.path.join(ROOT, "include"), src, "-o", out,
                        "-L", LIB, "-lhorizonator", "-lm", "-Wl,-rpath,$ORIGIN/../lib"], check=True)
    return out


if __name__ == "__main__":
    force = "--force" in sys.argv
    print(build_library(force=force, verbose=True))
    print(build_synth(force=force))
    print(build_cli(force=force))
