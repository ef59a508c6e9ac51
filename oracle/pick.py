"""Numpy restatement of the ground point of a rendered pixel (horizonator_pick_batch*, include/horizonator-batch.h),
used only by the tests: given a view, a pixel and the number of the triangle drawn there, the triangle's window
positions are recomputed from the same float inputs as the renderer's (its float eye, axis tables and projection) and
the ground point interpolated from them in double, operation for operation as k_pick does it.

The vertex arithmetic is oracle/vertex.py's; pass atan=device_atan(lib) to evaluate the renderer's own angle functions
on the GPU, which makes the window positions bit-identical to the renderer's."""
import math

import numpy as np

from oracle.vertex import (CELL_MASK, LOD_SHIFT, TILE_CELLS, axis, device_atan, eye, numpy_atan, project,  # noqa: F401
                           vertices, window)

F = np.float32
SKY = 0xFFFFFFFF


def window_positions(tri, mosaic, N, eye_, win, W, H, copy=0, curvature=0.0, atan=numpy_atan, cpd=1200):
    """the triangle's gl_Position.x (xn) and unsnapped float32 window positions (xw, yw), its vertices (vj, vi),
    heights z and metres e, n (k_prepare's axis tables, hz_project, the viewport transform: oracle/vertex.py)"""
    vci, vcj, vz, cos_lat = eye_
    vj, vi = vertices(tri, N)
    e = axis(vi, vci, cpd, cos_lat)
    n = axis(vj, vcj, cpd)
    z = np.array([F(mosaic[a, b]) for a, b in zip(vj, vi)], F)
    xn, xw, yw = project(e, n, z, eye_, win, W, H, F(curvature), atan, copy)
    return xn, xw, yw, vj, vi, z, e, n


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
