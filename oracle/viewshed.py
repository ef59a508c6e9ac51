"""oracle/viewshed.py -- TEST INFRASTRUCTURE.  ctypes access to the viewshed oracle (viewshed_oracle.c).

Only tests/ and tools/ may import this.  The library is compiled on first use with the oracle's own flags (one IEEE
rounding per source operator) and linked to liboracle.so, whose public functions supply the heights and the eye.

    vs = ViewshedOracle(oracle)          # an oracle.binding.Oracle; its current eye (oracle_move) is used
    words = vs.words(target_height=1.7)  # (N, (N+31)//32) uint32, as horizonator-batch.h lays out a mask
    mask = vs.mask(exact=True)           # (N, N) bool; exact=True: brute-force line of sight instead of R2
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from .binding import ORACLE_SO, Oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "viewshed_oracle.c")
# the system gcc: the image's default CC is a wrapper without libgomp (oracle/Makefile)
HOSTCC = os.environ.get("HOSTCC", "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc")
CFLAGS = ["-O2", "-g", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra", "-std=gnu11"]

_LIB = None


def _build():
    """viewshed_oracle.so next to its source, or in the temporary directory where oracle/ is not writable."""
    Oracle.lib()                                          # liboracle.so exists from here on
    for d in (HERE, os.path.join(tempfile.gettempdir(), "hz_viewshed_oracle_%d" % os.getuid())):
        out = os.path.join(d, "viewshed_oracle.so")
        try:
            os.makedirs(d, exist_ok=True)
            if not os.access(d, os.W_OK):
                continue
            if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(SRC), os.path.getmtime(ORACLE_SO)):
                tmp = out + ".%d.tmp" % os.getpid()
                subprocess.run([HOSTCC] + CFLAGS + ["-shared", "-I", HERE, "-o", tmp, SRC, ORACLE_SO,
                                                    "-Wl,-rpath," + HERE, "-lm"], check=True)
                os.replace(tmp, out)
            return out
        except PermissionError:
            continue
    raise RuntimeError("no writable directory for viewshed_oracle.so")


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(_build())
        vp, f, i, b = C.c_void_p, C.c_float, C.c_int, C.c_bool
        L.vs_oracle_mosaic.argtypes = [vp, vp]
        L.vs_oracle_mosaic.restype = None
        for name in ("vs_oracle_r2", "vs_oracle_exact"):
            getattr(L, name).argtypes = [vp, vp, f, f, i, vp]
            getattr(L, name).restype = b
        _LIB = L
    return _LIB


def unpack_mask(words):
    """(..., N, W32) uint32 viewshed words -> (..., N, N) bool (cell i of row j = bit i & 31 of word [j][i >> 5])."""
    words = np.ascontiguousarray(words, dtype="<u4")
    n = words.shape[-2]
    bits = np.unpackbits(words.view(np.uint8), axis=-1, bitorder="little")
    return bits[..., :n].astype(bool)


class ViewshedOracle:
    """Viewsheds of `oracle`'s current eye over its DEM square.  curvature: the coefficient of the apparent height drop
    (as Oracle.set_curvature / horizonator_set_earth_curvature; 0 = flat earth); threads: OpenMP threads."""

    def __init__(self, oracle, threads=None):
        self.o = oracle
        self.threads = threads or os.cpu_count() or 1
        n = 2 * oracle.dem_geometry()["radius_cells"]
        self.heights = np.empty((n, n), np.int16)
        lib().vs_oracle_mosaic(oracle.h, self.heights.ctypes.data)

    def words(self, target_height=0., exact=False, curvature=0.):
        n = self.heights.shape[0]
        out = np.zeros((n, (n + 31) // 32), np.uint32)
        fn = lib().vs_oracle_exact if exact else lib().vs_oracle_r2
        if not fn(self.o.h, self.heights.ctypes.data, curvature, target_height, self.threads, out.ctypes.data):
            raise ValueError("the eye is not inside the loaded square")
        return out

    def mask(self, target_height=0., exact=False, curvature=0.):
        return unpack_mask(self.words(target_height, exact, curvature))
