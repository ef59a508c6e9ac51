"""Numpy restatement of the ground point of a rendered pixel (horizonator_pick_batch*, include/horizonator-batch.h),
used only by the tests: given a view, a pixel and the number of the triangle drawn there, the triangle's window
positions are recomputed from the same float inputs as the renderer's (its float eye, axis tables and projection) and
the ground point interpolated from them in double, operation for operation as k_pick does it.

The renderer's fp32 angle functions are approximations of their own (csrc/hz_math.cuh); pass atan=device_atan(lib) to
evaluate them on the GPU through horizonator_debug_device_math(), which makes the window positions bit-identical to
the renderer's.  The default, numpy's float32 arctan2, is within a few ulp of them."""
import ctypes as C
import ctypes.util
import math

import numpy as np

F = np.float32
PI_F = F(3.14159265358979)           # hz_math.cuh HZ_PI_F
REARTH_F = F(6371000.0)
LOD_SHIFT, CELL_MASK, TILE_CELLS = 29, 0x1FFFFFFF, 32
SKY = 0xFFFFFFFF

_libm = C.CDLL(ctypes.util.find_library("m"))
_libm.cosf.restype, _libm.cosf.argtypes = C.c_float, [C.c_float]


def numpy_atan(e, n, h, d2):
    """float32 (azimuth atan2(e, n), elevation atan(h / sqrt(d2))) of arrays"""
    return np.arctan2(e, n).astype(F), np.arctan2(h, np.sqrt(d2)).astype(F)


def device_atan(lib):
    """the renderer's own hz_atan2_az / hz_atan_el, evaluated on the current CUDA device"""
    def f(e, n, h, d2):
        e, n, h, d2 = (np.ascontiguousarray(a, F) for a in (e, n, h, d2))
        az, el = np.empty_like(e), np.empty_like(e)
        p = lambda a: a.ctypes.data
        assert lib.horizonator_debug_device_math(len(e), p(e), p(n), p(h), p(d2), p(az), p(el))
        return az, el
    return f


def eye(dem, mosaic, lat, lon, viewer_z=-1.0):
    """(viewer_cell_i, viewer_cell_j, viewer_z, cos_viewer_lat) in float32 as horizonator_move() computes them
    (lib:765-799).  dem: (origin lon, origin lat, cell_i, cell_j, cells_per_deg); mosaic: [j][i] heights."""
    lon_deg, lat_deg, ci, cj, cpd = dem
    vci = F(F(F(lon) - F(lon_deg)) * F(cpd)) - F(ci)
    vcj = F(F(F(lat) - F(lat_deg)) * F(cpd)) - F(cj)
    if viewer_z < 0:
        i0, j0 = int(math.floor(vci)), int(math.floor(vcj))
        viewer_z = F(float(max(mosaic[j0, i0], mosaic[j0, i0 + 1], mosaic[j0 + 1, i0], mosaic[j0 + 1, i0 + 1])) + 1.0)
    return vci, vcj, F(viewer_z), F(_libm.cosf(float(F(float(F(lat)) * math.pi / 180.0))))


def window(az_deg0, az_deg1, W, H, seam_wrap=False):
    """(az_center, az_ndc_per_rad, aspect, seam_period) in float32 as the host fills them (vertex.glsl:139-150)"""
    r0 = F(F(az_deg0) * F(0.017453292519943295))
    r1 = F(F(az_deg1) * F(0.017453292519943295))
    d = F(F(F(r1 - r0) - PI_F) / F(F(2.0) * PI_F))
    r1 = F(F(F(F(d - F(np.rint(d))) * F(2.0)) * PI_F) + PI_F) + r0
    per_rad = F(F(2.0) / F(r1 - r0))
    return F(F(r0 + r1) / F(2.0)), per_rad, F(F(W) / F(H)), F(F(per_rad * F(2.0)) * PI_F) if seam_wrap else F(0.0)


def vertices(tri, N):
    """triangle number (level of detail in bits [30:29]) -> its vertices' rows vj and columns vi (lib:496-508)"""
    s = 1 << (tri >> LOD_SHIFT)
    cell = (tri & CELL_MASK) >> 1
    j, i = cell // (N - 1), cell % (N - 1)
    if tri & 1 == 0:
        return [j, j + s, j + s], [i, i + s, i]
    return [j, j, j + s], [i, i + s, i + s]


def window_positions(tri, mosaic, N, eye_, win, W, H, copy=0, curvature=0.0, atan=numpy_atan, cpd=1200):
    """the triangle's gl_Position.x (xn) and unsnapped float32 window positions (xw, yw), its vertices (vj, vi),
    heights z and metres e, n (k_prepare's axis tables, hz_project, the viewport transform: vertex.glsl:128-153)"""
    vci, vcj, vz, cos_lat = eye_
    center, per_rad, aspect, period = win
    vj, vi = vertices(tri, N)
    dpc = F(F(1.0) / F(cpd))
    e = np.array([F(F(F(F(F(F(c) - vci) * dpc) * REARTH_F) * PI_F) / F(180.0)) * cos_lat for c in vi], F)
    n = np.array([F(F(F(F(F(c) - vcj) * dpc) * REARTH_F) * PI_F) / F(180.0) for c in vj], F)
    z = np.array([F(mosaic[a, b]) for a, b in zip(vj, vi)], F)
    d2 = (e * e + n * n).astype(F)
    h = ((z - vz) - (F(curvature) * d2)).astype(F)
    az, el = atan(e, n, h, d2)
    t = ((az - center) * F(0.15915494309189535)).astype(F)
    az = ((((t - np.rint(t)).astype(F) * F(2.0)) * PI_F) + center).astype(F)
    xn = ((az - center) * per_rad).astype(F)
    yn = ((el * aspect) * per_rad).astype(F)
    if copy >= 1:
        xn = np.where(xn < 0, xn + period, xn).astype(F)
    if copy == 2:
        xn = (xn - period).astype(F)
    halfW, halfH = F(F(0.5) * F(W)), F(F(0.5) * F(H))
    return xn, (xn * halfW + halfW).astype(F), (yn * halfH + halfH).astype(F), vj, vi, z, e, n


def weights(cx, cy, xw, yw):
    """barycentric weights (b0, b1, b2) of (cx, cy), in double from the float positions, not clamped"""
    x0, x1, x2 = (float(v) for v in xw)
    y0, y1, y2 = (float(v) for v in yw)
    d = (x1 - x0) * (y2 - y0) - (x2 - x0) * (y1 - y0)
    b1 = ((cx - x0) * (y2 - y0) - (x2 - x0) * (cy - y0)) / d
    b2 = ((x1 - x0) * (cy - y0) - (cx - x0) * (y1 - y0)) / d
    return 1.0 - b1 - b2, b1, b2


def point(b, vj, vi, z, e, n, dem):
    """(lat, lon, ele_m, distance_m) of weights b over the vertices: lat / lon by the DEM geometry of the header"""
    lon_deg, lat_deg, ci, cj, cpd = dem
    S = lambda a: b[0] * float(a[0]) + b[1] * float(a[1]) + b[2] * float(a[2])
    i, j, ge, gn = S(vi), S(vj), S(e), S(n)
    return (float(lat_deg) + (float(cj) + j) / float(cpd), float(lon_deg) + (float(ci) + i) / float(cpd),
            float(F(S(z))), float(F(math.sqrt(ge * ge + gn * gn))))


def ground(tri, x, y, mosaic, N, eye_, win, W, H, dem, curvature=0.0, atan=numpy_atan):
    """(lat, lon, ele_m, distance_m) of pixel (x, y) (image row y, 0 = top) showing triangle `tri`"""
    cx, cy = x + 0.5, (H - 1 - y) + 0.5
    kw = dict(curvature=curvature, atan=atan, cpd=dem[4])
    xn, xw, yw, vj, vi, z, e, n = window_positions(tri, mosaic, N, eye_, win, W, H, 0, **kw)
    if win[3] > 0 and float(F(xn.max() - xn.min())) > 0.5:          # too wide: with the seam wrap, one of its copies
        xn, xw, yw, vj, vi, z, e, n = window_positions(tri, mosaic, N, eye_, win, W, H, 1, **kw)
        if not (float(xw.min()) <= cx <= float(xw.max())):
            xn, xw, yw, vj, vi, z, e, n = window_positions(tri, mosaic, N, eye_, win, W, H, 2, **kw)
    return point(weights(cx, cy, xw, yw), vj, vi, z, e, n, dem)
