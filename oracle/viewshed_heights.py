"""oracle/viewshed_heights.py -- TEST INFRASTRUCTURE.  ctypes access to the viewshed heights oracle
(viewshed_heights_oracle.c, vs_oracle_r2_heights).

Only tests/ and tools/ may import this.  The library is compiled on first use with the viewshed oracle's flags (one IEEE
rounding per source operator) and linked to liboracle.so, like oracle/viewshed.py's.

    vs = ViewshedOracle(oracle)          # oracle.viewshed: an Oracle's current eye and its square's terrain
    h = r2_heights(vs, curvature=0.)     # (N, N) float32: the least height above the ground at which the eye sees
                                         # each vertex under R2 (+inf where no ray decides it)
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from .binding import ORACLE_SO, Oracle
from .viewshed import CFLAGS, HOSTCC, HERE, SRC as VS_SRC

SRC = os.path.join(HERE, "viewshed_heights_oracle.c")

_LIB = None


def _build():
    """viewshed_heights_oracle.so next to its source, or in the temporary directory where oracle/ is not writable."""
    Oracle.lib()                                          # liboracle.so exists from here on
    deps = (SRC, VS_SRC, ORACLE_SO)
    for d in (HERE, os.path.join(tempfile.gettempdir(), "hz_viewshed_oracle_%d" % os.getuid())):
        out = os.path.join(d, "viewshed_heights_oracle.so")
        try:
            os.makedirs(d, exist_ok=True)
            if not os.access(d, os.W_OK):
                continue
            if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(p) for p in deps):
                tmp = out + ".%d.tmp" % os.getpid()
                subprocess.run([HOSTCC] + CFLAGS + ["-shared", "-I", HERE, "-o", tmp, SRC, ORACLE_SO,
                                                    "-Wl,-rpath," + HERE, "-lm"], check=True)
                os.replace(tmp, out)
            return out
        except PermissionError:
            continue
    raise RuntimeError("no writable directory for viewshed_heights_oracle.so")


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(_build())
        L.vs_oracle_r2_heights.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_void_p]
        L.vs_oracle_r2_heights.restype = C.c_bool
        _LIB = L
    return _LIB


def r2_heights(vs, curvature=0.):
    """(N, N) float32 [j north][i east] for the current eye of `vs` (an oracle.viewshed.ViewshedOracle, whose terrain
    and thread count it uses): how far above the ground each vertex must rise for the eye to see it under R2
    (horizonator_viewshed_heights; +inf where no ray decides the vertex)"""
    n = vs.heights.shape[0]
    out = np.empty((n, n), np.float32)
    if not lib().vs_oracle_r2_heights(vs.o.h, vs.heights.ctypes.data, curvature, vs.threads, out.ctypes.data):
        raise ValueError("the eye is not inside the loaded square")
    return out
