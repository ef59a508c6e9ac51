"""Ground points of rendered pixels (horizonator_pick_batch*, include/horizonator-batch.h), checked without a GPU: the
ctypes mirrors of horizonator_pixel_t / horizonator_ground_t against a compiled probe of the header, and the host
restatement (oracle/pick.py, which the GPU tests compare the kernel with) on hand-made triangles, including the DEM
geometry of its latitudes and longitudes against the library's host horizonator_project()."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import pick as op

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GCC = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"

PROBE = r"""
#include <stddef.h>
#include <stdio.h>
#include "horizonator-batch.h"
int main(void)
{
    printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(horizonator_pixel_t), offsetof(horizonator_pixel_t, x),
           offsetof(horizonator_pixel_t, y), sizeof(horizonator_ground_t), offsetof(horizonator_ground_t, lat),
           offsetof(horizonator_ground_t, lon), offsetof(horizonator_ground_t, ele_m),
           offsetof(horizonator_ground_t, range_m), offsetof(horizonator_ground_t, distance_m),
           offsetof(horizonator_ground_t, triangle));
    return 0;
}
"""


def test_ctypes_mirrors_match_the_header(tmp_path):
    import horizonator_b200 as hz
    src, exe = tmp_path / "probe.c", tmp_path / "probe"
    src.write_text(PROBE)
    subprocess.run([GCC, "-std=gnu99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [8, 0, 4, 32, 0, 8, 16, 20, 24, 28]
    assert C.sizeof(hz.pixel_t) == 8 and [hz.pixel_t.x.offset, hz.pixel_t.y.offset] == [0, 4]
    assert C.sizeof(hz.ground_t) == 32
    names = ["lat", "lon", "ele_m", "range_m", "distance_m", "triangle"]
    assert [getattr(hz.ground_t, k).offset for k in names] == got[4:]
    assert hz.GROUND_DTYPE.itemsize == 32 and [hz.GROUND_DTYPE.fields[k][1] for k in names] == got[4:]


# ---- hand-made triangles

N = 2400
DEM = (-118, 34, 600, 840, 1200)          # origin lon, lat, cell i, cell j, cells per degree


def _mosaic(seed=3):
    rs = np.random.default_rng(seed)
    return rs.integers(200, 3000, (N + 16, N + 16)).astype(np.int16)


def test_vertices_follow_the_reference_numbering_and_the_level_bits():
    for half in (0, 1):
        tri = 2 * (7 * (N - 1) + 11) + half
        vj, vi = op.vertices(tri, N)
        assert (vj[0], vi[0]) == (7, 11)
        assert (vj, vi) == (([7, 8, 8], [11, 12, 11]) if half == 0 else ([7, 7, 8], [11, 12, 12]))
        vj2, vi2 = op.vertices(tri | (2 << op.LOD_SHIFT), N)
        assert (vj2, vi2) == (([7, 11, 11], [11, 15, 11]) if half == 0 else ([7, 7, 11], [11, 15, 15]))


@pytest.mark.parametrize("b,k", [((1.0, 0.0, 0.0), 0), ((0.0, 1.0, 0.0), 1), ((0.0, 0.0, 1.0), 2)])
def test_a_vertex_weight_gives_that_vertex(b, k):
    mosaic = _mosaic()
    tri = 2 * (1300 * (N - 1) + 977) + 1
    eye = op.eye(DEM, mosaic, 34.0 + (840 + 1200.3) / 1200, -118.0 + (600 + 1201.7) / 1200)
    win = op.window(-180.0, 179.9, 3600, 600)
    xn, xw, yw, vj, vi, z, e, n = op.window_positions(tri, mosaic, N, eye, win, 3600, 600)
    lat, lon, ele, dist = op.point(b, vj, vi, z, e, n, DEM)
    assert lat == DEM[1] + (DEM[3] + vj[k]) / DEM[4] and lon == DEM[0] + (DEM[2] + vi[k]) / DEM[4]
    assert ele == float(z[k]) and dist == float(np.float32(math.hypot(float(e[k]), float(n[k]))))


def test_vertex_lat_lon_agree_with_horizonator_project():
    """The DEM geometry of the header, fed to horizonator_project(), puts a vertex where the renderer's metres east and
    north of the eye (in double) put it: within 1e-9 pixel."""
    import horizonator_b200 as hz
    mosaic = _mosaic()
    W, H, az0, az1 = 3600, 600, -180.0, 179.9
    lat0, lon0 = 34.0 + (840 + 1200.3) / 1200, -118.0 + (600 + 1201.7) / 1200
    ele0 = 1800.0
    cos_lat = math.cos(lat0 * math.pi / 180.)
    vci, vcj = (lon0 - DEM[0]) * DEM[4] - DEM[2], (lat0 - DEM[1]) * DEM[4] - DEM[3]
    x, y, r = C.c_double(), C.c_double(), C.c_double()
    rs = np.random.default_rng(5)
    for k in range(50):
        tri = 2 * (int(rs.integers(0, N - 1)) * (N - 1) + int(rs.integers(0, N - 1))) + k % 2
        vj, vi = op.vertices(tri, N)
        z = float(mosaic[vj[0], vi[0]])
        lat, lon, ele, _ = op.point((1.0, 0.0, 0.0), vj, vi, [z, 0, 0], [0, 0, 0], [0, 0, 0], DEM)
        if not hz.lib.horizonator_project(C.byref(x), C.byref(y), C.byref(r), lat0, cos_lat, lon0, ele0, lat, lon, ele,
                                          az0 * math.pi / 180., az1 * math.pi / 180., W, H):
            continue
        # the renderer's vertex (vertex.glsl:128-153) in double
        e = (vi[0] - vci) / DEM[4] * 6371000.0 * math.pi / 180. * cos_lat
        n = (vj[0] - vcj) / DEM[4] * 6371000.0 * math.pi / 180.
        per_rad = 2.0 / ((az1 - az0) * math.pi / 180.)
        center = (az0 + az1) / 2. * math.pi / 180.
        az = math.atan2(e, n)
        az = center + math.remainder(az - center, 2 * math.pi)
        want_x = ((az - center) * per_rad + 1.) / 2. * W - 0.5
        el = math.atan2(z - ele0, math.hypot(e, n)) * (W / H) * per_rad
        want_y = (-el + 1.) / 2. * H - 0.5
        assert abs(x.value - want_x) < 1e-9 and abs(y.value - want_y) < 1e-9, (k, x.value - want_x, y.value - want_y)


def test_weights_of_the_centroid_and_outside_points():
    xw, yw = np.array([10.25, 14.75, 11.5], np.float32), np.array([3.5, 4.0, 9.25], np.float32)
    cx, cy = float(sum(map(float, xw))) / 3, float(sum(map(float, yw))) / 3
    b = op.weights(cx, cy, xw, yw)
    assert max(abs(v - 1 / 3) for v in b) < 1e-12 and abs(sum(b) - 1.0) < 1e-15
    # outside the triangle: negative weights, not clamped; interpolation reproduces the point
    b = op.weights(20.0, 0.0, xw, yw)
    assert min(b) < 0
    assert abs(sum(w * float(v) for w, v in zip(b, xw)) - 20.0) < 1e-12
    assert abs(sum(w * float(v) for w, v in zip(b, yw)) - 0.0) < 1e-12


def test_ground_of_a_pixel_inside_a_triangle_lies_inside_it():
    mosaic = _mosaic()
    W, H = 1200, 300
    eye = op.eye(DEM, mosaic, 34.0 + (840 + 1200.3) / 1200, -118.0 + (600 + 1201.7) / 1200)
    win = op.window(-30.0, 30.0, W, H)
    # a triangle north of the eye, 30 cells away
    tri = 2 * (1230 * (N - 1) + 1201)
    xn, xw, yw, vj, vi, z, e, n = op.window_positions(tri, mosaic, N, eye, win, W, H)
    cx, cy = float(np.mean(xw)), float(np.mean(yw))
    x, y = int(math.floor(cx)), H - 1 - int(math.floor(cy))
    lat, lon, ele, dist = op.ground(tri, x, y, mosaic, N, eye, win, W, H, DEM)
    j = (lat - DEM[1]) * DEM[4] - DEM[3]
    i = (lon - DEM[0]) * DEM[4] - DEM[2]
    assert min(vj) - 1e-6 <= j <= max(vj) + 1e-6 and min(vi) - 1e-6 <= i <= max(vi) + 1e-6
    assert float(z.min()) - 1e-3 <= ele <= float(z.max()) + 1e-3
    assert min(math.hypot(float(a), float(b)) for a, b in zip(e, n)) - 1 <= dist <= max(
        math.hypot(float(a), float(b)) for a, b in zip(e, n)) + 1
