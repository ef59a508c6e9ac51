"""Numpy restatement of the renderer's vertex stage, used only by the tests: k_prepare's axis tables, hz_project and
hz_depth_shade (csrc/hz_kernels.cu), the viewport transform and the seam copies, in float32 operator by operator as
the kernels evaluate them (-fmad=false: every operator one IEEE rounding).  Also the host's eye and window scalars and
the level-of-detail rule of enqueue_views() (csrc/hz_api.cpp), for the exact reference (tests/test_exact_reference.py,
tests/test_gpu_exact.py) and the ground points (oracle/pick.py).

The renderer's fp32 angle functions are approximations of their own (csrc/hz_math.cuh); pass atan=device_atan(lib) to
evaluate them on the GPU through horizonator_debug_device_math(), which makes every vertex bit-identical to the
renderer's.  The default, numpy's float32 arctan2, is within a few ulp of them."""
import ctypes as C
import ctypes.util
import math

import numpy as np

F = np.float32
PI_F = F(3.14159265358979)           # hz_math.cuh HZ_PI_F
REARTH_F = F(6371000.0)
INV_2PI_F = F(0.15915494309189535)   # hz_project's rounded 1/(2 pi)
LOD_SHIFT, CELL_MASK, TILE_CELLS = 29, 0x1FFFFFFF, 32
NEAR_RINGS, MAX_LOD = 2, 2           # hz_api.cpp NEAR_RINGS, hz_device.h HZ_MAX_LOD
VTX = np.dtype([("x_ndc", F), ("xw", F), ("yw", F), ("zw", F), ("r", F)])    # glp_vtx_t (oracle/gl_pipeline.h)

_libm = C.CDLL(ctypes.util.find_library("m"))
_libm.cosf.restype, _libm.cosf.argtypes = C.c_float, [C.c_float]


def numpy_atan(e, n, h, d2):
    """float32 (azimuth atan2(e, n), elevation atan(h / sqrt(d2))) of arrays"""
    return np.arctan2(e, n).astype(F), np.arctan2(h, np.sqrt(d2)).astype(F)


def device_atan(lib, chunk=1 << 24):
    """the renderer's own hz_atan2_az / hz_atan_el, evaluated on the current CUDA device, `chunk` values per call"""
    def f(e, n, h, d2):
        e, n, h, d2 = (np.ascontiguousarray(a, F).ravel() for a in (e, n, h, d2))
        az, el = np.empty_like(e), np.empty_like(e)
        for s in range(0, len(e), chunk):
            p = lambda a: a[s:].ctypes.data
            assert lib.horizonator_debug_device_math(min(chunk, len(e) - s), p(e), p(n), p(h), p(d2), p(az), p(el))
        return az, el
    return f


def eye(dem, mosaic, lat, lon, viewer_z=-1.0):
    """(viewer_cell_i, viewer_cell_j, viewer_z, cos_viewer_lat) in float32 as horizonator_move() computes them
    (lib:765-799).  dem: (origin lon, origin lat, cell_i, cell_j, cells_per_deg); mosaic: [j][i] heights.  The
    automatic eye height reads the mosaic: pass viewer_z for an eye on or beyond its last row or column."""
    lon_deg, lat_deg, ci, cj, cpd = dem
    vci = F(F(F(lon) - F(lon_deg)) * F(cpd)) - F(ci)
    vcj = F(F(F(lat) - F(lat_deg)) * F(cpd)) - F(cj)
    if viewer_z < 0:
        i0, j0 = int(math.floor(vci)), int(math.floor(vcj))
        assert 0 <= i0 < mosaic.shape[1] - 1 and 0 <= j0 < mosaic.shape[0] - 1, "eye outside the mosaic: give viewer_z"
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


def curvature(on=True, refraction=0.13):
    """the coefficient horizonator_set_earth_curvature() stores: (1 - refraction) / (2 Rearth), float"""
    return F(F(F(1.0) - F(refraction)) / F(F(2.0) * REARTH_F)) if on else F(0.0)


def axis(c, vc, cpd, cos_lat=None):
    """k_prepare's e_tab (with cos_lat) or n_tab for the columns / rows c: (c - vc) * DEG_PER_CELL * Rearth * pi / 180
    [* cos_lat] (vertex.glsl:128-130)"""
    dpc = F(F(1.0) / F(cpd))
    t = ((((np.asarray(c).astype(F) - vc) * dpc) * REARTH_F) * PI_F) / F(180.0)
    return (t * cos_lat if cos_lat is not None else t).astype(F)


def project(e, n, z, eye_, win, W, H, curv=F(0.0), atan=numpy_atan, copy=0):
    """hz_project and the viewport transform of vertices at e, n metres from the eye with heights z:
    (gl_Position.x, window x, window y), float32 arrays.  copy 1 / 2: the seam copies of hz_tri_project."""
    vz = eye_[2]
    center, per_rad, aspect, period = win
    d2 = (e * e + n * n).astype(F)
    h = ((z - vz) - (F(curv) * d2)).astype(F)
    az, el = atan(e, n, h, d2)
    az, el = az.reshape(np.shape(e)), el.reshape(np.shape(e))
    t = ((az - center) * INV_2PI_F).astype(F)
    az = ((((t - np.rint(t)).astype(F) * F(2.0)) * PI_F) + center).astype(F)
    xn = ((az - center) * per_rad).astype(F)
    yn = ((el * aspect) * per_rad).astype(F)
    if copy >= 1:
        xn = np.where(xn < 0, xn + period, xn).astype(F)
    if copy == 2:
        xn = (xn - period).astype(F)
    halfW, halfH = F(F(0.5) * F(W)), F(F(0.5) * F(H))
    return xn, (xn * halfW + halfW).astype(F), (yn * halfH + halfH).astype(F)


def depth_shade(e, n, z, vz, zext, curv=F(0.0)):
    """hz_depth_shade: window depth zw and red channel r, float32 arrays.  zext: (znear, zfar, znear_color, zfar_color)"""
    znear, zfar, znc, zfc = (F(v) for v in zext)
    d2 = (e * e + n * n).astype(F)
    h = ((z - vz) - (F(curv) * d2)).astype(F)
    dne = np.sqrt(d2)
    ln = np.sqrt((d2 + h * h).astype(F))
    zn = ((((ln - znear) / F(zfar - znear)) * F(2.0)) - F(1.0)).astype(F)
    zw = ((zn * F(0.5)) + F(0.5)).astype(F)
    r = np.maximum(np.minimum(((dne - znc) / F(zfc - znc)).astype(F), F(1.0)), F(0.0)).astype(F)
    return zw, r


def grid(mosaic, N, eye_, win, W, H, zext, cpd, curv=F(0.0), atan=numpy_atan, rows=256):
    """The vertex stage of every vertex of the N x N mesh, as glp_vtx_t records [j * N + i] (oracle/gl_pipeline.h),
    computed `rows` rows at a time"""
    vci, vcj, vz, cos_lat = eye_
    e_tab = axis(np.arange(N), vci, cpd, cos_lat)
    n_tab = axis(np.arange(N), vcj, cpd)
    out = np.empty(N * N, VTX)
    for j0 in range(0, N, rows):
        j1 = min(N, j0 + rows)
        e = np.broadcast_to(e_tab, (j1 - j0, N))
        n = np.broadcast_to(n_tab[j0:j1, None], (j1 - j0, N))
        z = mosaic[j0:j1, :N].astype(F)
        o = out[j0 * N:j1 * N].reshape(j1 - j0, N)
        o["x_ndc"], o["xw"], o["yw"] = project(e, n, z, eye_, win, W, H, curv, atan)
        o["zw"], o["r"] = depth_shade(e, n, z, vz, zext, curv)
    return out


def n_tiles(N):
    """tiles of TILE_CELLS x TILE_CELLS cells per side of the mesh of N x N vertices"""
    return (N - 1 + TILE_CELLS - 1) // TILE_CELLS


def lod_from(per_rad, W, lod_pixels):
    """enqueue_views(): the first ring of tiles drawn at each level (lod_from[0] = 0); lod_pixels 0 = off"""
    out = [0] + [1 << 30] * MAX_LOD
    if lod_pixels > 0:
        k_px = abs(float(F(per_rad))) * 0.5 * float(W) / float(TILE_CELLS)
        for l in range(1, MAX_LOD + 1):
            r = math.ceil(k_px * float(1 << l) / float(F(lod_pixels))) + 1.0
            out[l] = 2 if r < 2.0 else ((1 << 30) if r > 1e9 else int(r))
    return out


def tile_levels(N, eye_, per_rad, W, lod_pixels):
    """int8 [tj][ti]: the level of detail each tile is drawn at.  Ring r of a tile = its Chebyshev distance in tiles
    from the eye's tile (clamped to the mesh); rings up to NEAR_RINGS (the near pass) are level 0, a ring r beyond
    has level max{l : r >= lod_from[l]}."""
    nt = n_tiles(N)
    tc = F(TILE_CELLS)
    ti = min(max(int(np.floor(F(eye_[0]) / tc)), 0), nt - 1)
    tj = min(max(int(np.floor(F(eye_[1]) / tc)), 0), nt - 1)
    a = np.arange(nt)
    ring = np.maximum(np.abs(a[:, None] - tj), np.abs(a[None, :] - ti))
    lv = np.zeros((nt, nt), np.int8)
    for l, r0 in enumerate(lod_from(per_rad, W, lod_pixels)):
        if l > 0:
            lv[(ring > NEAR_RINGS) & (ring >= r0)] = l
    return lv


def vertices(tri, N):
    """triangle number (level of detail in bits [30:29]) -> its vertices' rows vj and columns vi (lib:496-508)"""
    s = 1 << (tri >> LOD_SHIFT)
    cell = (tri & CELL_MASK) >> 1
    j, i = cell // (N - 1), cell % (N - 1)
    if tri & 1 == 0:
        return [j, j + s, j + s], [i, i + s, i]
    return [j, j, j + s], [i, i + s, i + s]
