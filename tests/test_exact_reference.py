"""The exact reference of the renderer, checked without a GPU: the key rasteriser of the oracle (glp_draw_keys(),
oracle/gl_pipeline.c), which draws every triangle of a vertex stage without any culling into per-pixel visibility keys
by the oracle's own rules F2-F8, and the level-of-detail triangle set (oracle/vertex.py).  tests/test_gpu_exact.py
compares the CUDA renderer with it bit for bit."""
import os

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON
from oracle import binding
from oracle import vertex as ov

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _golden_scenes():
    return sorted(f[len("render_"):-len(".npz")] for f in os.listdir(GOLDEN) if f.startswith("render_"))


def _keys_of_oracle(o, W, H, az0, az1, zn, zf, threads=None, **kw):
    vtx, period = o.vertex_stage(az0, az1, znear=zn, zfar=zf, **kw)
    N = 2 * o.dem_geometry()["radius_cells"]
    return binding.draw_keys(vtx, N, W, H, period, threads=threads), vtx, N


@pytest.mark.parametrize("name", _golden_scenes())
def test_keys_of_the_oracle_vertex_stage_give_the_golden_render(tiles_c1, name):
    """Fed the oracle's own vertex stage, the unculled key rasteriser with its min-merge and the oracle's read-back
    give the recorded render of the reference bit for bit: every triangle enumerated, the merge equal to GL_LESS in
    draw order, the read-back shared."""
    g = np.load(os.path.join(GOLDEN, "render_%s.npz" % name))
    W, H, R, az0, az1, zn, zf, znc, zfc, lat, lon = g["params"]
    W, H, R = int(W), int(H), int(R)
    o = binding.Oracle(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    kw = {} if lat <= -1000. else dict(lat=float(lat), lon=float(lon))
    keys, _, _ = _keys_of_oracle(o, W, H, float(az0), float(az1), float(zn), float(zf), threads=3,
                                 znear_color=float(znc), zfar_color=float(zfc), **kw)
    img, rng = binding.read_keys(keys, float(az0), float(az1), float(zn), float(zf))
    assert np.array_equal(img, g["image"])
    assert np.array_equal(rng.view(np.uint32), g["ranges"].view(np.uint32))


@pytest.mark.parametrize("mode", ["seam_wrap", "curvature"])
def test_keys_equal_the_oracle_render_in_the_opt_in_modes(tiles_c1, mode):
    W, H, R, az0, az1 = 360, 75, 120, -180.05, 179.95
    o = binding.Oracle(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R, threads=4)
    if mode == "seam_wrap":
        o.set_seam_wrap(True)
    else:
        o.set_curvature(float(ov.curvature()))
    want = o.render(az0, az1, znear=50., zfar=100000.)
    keys, _, _ = _keys_of_oracle(o, W, H, az0, az1, 50., 100000.)
    img, rng = binding.read_keys(keys, az0, az1, 50., 100000.)
    assert np.array_equal(img, want[0]) and np.array_equal(rng.view(np.uint32), want[1].view(np.uint32))
    assert (rng > 0).mean() > 0.05


def _snap(a):
    """F2 on float32 window coordinates"""
    t = np.asarray(a, np.float32) * np.float32(256.0)
    return np.where(np.abs(t) < np.float32(8388608.0), np.floor(t + np.float32(0.5)), t).astype(np.int64)


def _covers(X, Y, px, py):
    """F3/F4 on snapped positions X, Y (..., 3) for pixel centres (px, py): front-facing and inside by the fill rule"""
    Px, Py = px * 256 + 128, py * 256 + 128
    ok = (X[..., 1] - X[..., 0]) * (Y[..., 2] - Y[..., 0]) - (X[..., 2] - X[..., 0]) * (Y[..., 1] - Y[..., 0]) > 0
    for k in range(3):
        x0, y0, x1, y1 = X[..., k], Y[..., k], X[..., (k + 1) % 3], Y[..., (k + 1) % 3]
        dx, dy = x1 - x0, y1 - y0
        bias = np.where((dy < 0) | ((dy == 0) & (dx < 0)), 0, 1)
        ok = ok & (dx * (Py - y0) - dy * (Px - x0) >= bias)
    return ok


def _corners(tri, N):
    """vertex indices (j * N + i) of triangle numbers (level of detail in bits [30:29]), (..., 3)"""
    s = 1 << (tri >> ov.LOD_SHIFT).astype(np.int64)
    cell = (tri & ov.CELL_MASK).astype(np.int64) >> 1
    j, i = cell // (N - 1), cell % (N - 1)
    odd = (tri & 1).astype(bool)
    vj = np.stack([j, np.where(odd, j, j + s), j + s], -1)
    vi = np.stack([i, i + s, np.where(odd, i + s, i)], -1)
    return vj * N + vi


def test_the_winning_triangle_covers_the_pixel_centre(tiles_c1):
    W, H, R = 400, 100, 150
    o = binding.Oracle(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    keys, vtx, N = _keys_of_oracle(o, W, H, 20., 110., 100., 60000.)
    tri = binding.key_triangles(keys, N)[::-1]             # GL row order like the keys
    py, px = np.nonzero(tri != 0xFFFFFFFF)
    assert len(py) > 0.1 * W * H
    c = _corners(tri[py, px], N)
    assert _covers(_snap(vtx["xw"][c]), _snap(vtx["yw"][c]), px, py).all()
    # ... and its depth is that of the key: the plane of F6 at the pixel centre, quantised (F7)
    q = (keys[py, px] >> np.uint64(binding.KEY_Q_SHIFT)).astype(np.int64)
    assert (q < binding.Z24_MAX).all()


@pytest.mark.parametrize("threads", [1, 2, 3, 8])
def test_equal_depths_go_to_the_lowest_triangle_number(threads):
    """Hand-made ties: every cell of a 6 x 6 grid of vertices is drawn onto the same square (vertices of even and odd
    index alternate between two positions per axis, so every cell is the square itself, mirrored twice or not at all:
    mirrored once it faces away), all at the same depth.  Each pixel of the square holds the lowest-numbered
    triangle that covers it, whatever the number of threads, and its red channel."""
    N, W, H = 6, 24, 20
    j, i = np.divmod(np.arange(N * N), N)
    vtx = np.zeros(N * N, ov.VTX)
    vtx["xw"] = np.where(i % 2 == 0, 3.25, 19.5)
    vtx["yw"] = np.where(j % 2 == 0, 2.5, 17.75)
    vtx["x_ndc"] = 0.0                                                       # not "too wide" (geometry.glsl)
    vtx["zw"] = 0.5
    vtx["r"] = np.random.default_rng(1).uniform(0.1, 0.9, N * N).astype(np.float32)   # r8 differs between triangles
    keys = binding.draw_keys(vtx, N, W, H, threads=threads)
    tri = np.arange(2 * (N - 1) ** 2)
    c = _corners(tri, N)
    py, px = np.mgrid[0:H, 0:W]
    cov = _covers(_snap(vtx["xw"][c])[:, None, None], _snap(vtx["yw"][c])[:, None, None], px[None], py[None], )
    assert cov.any(0).sum() > 200 and (cov.sum(0) >= 8).any()               # many pixels with many candidates
    want = np.where(cov.any(0), np.where(cov, tri[:, None, None], 1 << 40).min(0), 0xFFFFFFFF)
    got = binding.key_triangles(keys, N)[::-1]
    assert np.array_equal(got, want)
    q = keys >> np.uint64(binding.KEY_Q_SHIFT)
    assert (q[cov.any(0)] == q[cov.any(0)].min()).all()                      # a tie everywhere
    # the red channel is the winner's own, not the least of the candidates'
    img, _ = binding.read_keys(keys, -45., 45., 100., 40000.)
    assert ((img[::-1][..., 2] != 0) == cov.any(0)).all()
    one = binding.draw_keys(vtx, N, W, H, threads=1)
    assert np.array_equal(keys, one)


@pytest.mark.parametrize("N", [2, 33, 70, 131])
@pytest.mark.parametrize("lod_pixels", [0.5, 1.0, 2.0])
def test_the_lod_set_tiles_the_ground_of_level_0(N, lod_pixels):
    """The cells the level-of-detail rule draws (a tile of level l: cells (j, i), multiples of s = 2^l, j, i <= N-1-s,
    each covering s x s cells of the dense grid) cover every cell of the dense grid exactly once, except the last
    (N - 1) mod s rows or columns of cells of a coarse tile at the mesh's far edges."""
    rs = np.random.default_rng(N)
    for _ in range(4):
        eye = (np.float32(rs.uniform(-40, N + 40)), np.float32(rs.uniform(-40, N + 40)))
        per_rad = np.float32(rs.uniform(0.2, 40.0))
        lv = ov.tile_levels(N, eye, per_rad, 3600, lod_pixels)
        T = ov.TILE_CELLS
        cover = np.zeros((N - 1, N - 1), np.int32)
        strip = np.zeros((N - 1, N - 1), bool)
        for tj in range(lv.shape[0]):
            for ti in range(lv.shape[1]):
                s = 1 << int(lv[tj, ti])
                for j in range(tj * T, min(tj * T + T, N - s), s):
                    for i in range(ti * T, min(ti * T + T, N - s), s):
                        cover[j:j + s, i:i + s] += 1
                last_j, last_i = min(tj * T + T, N - 1), min(ti * T + T, N - 1)
                e = (N - 1) % s
                if e and last_j == N - 1:
                    strip[N - 1 - e:, ti * T:last_i] = True
                if e and last_i == N - 1:
                    strip[tj * T:last_j, N - 1 - e:] = True
        assert (cover <= 1).all()
        assert (cover[~strip] == 1).all() and (cover[strip] == 0).all()


def test_lod_rule_follows_the_host():
    """lod_from[l] = max(2, ceil(k_px 2^l / lod_pixels) + 1), k_px = |az_ndc_per_rad| W / 64 in double; rings up
    to 2 are the near pass and stay at level 0"""
    per_rad = ov.window(-180.05, 179.95, 3600, 600)[1]
    k_px = abs(float(per_rad)) * 0.5 * 3600 / 32
    assert ov.lod_from(per_rad, 3600, 0.5) == [0, int(np.ceil(k_px * 2 / 0.5)) + 1, int(np.ceil(k_px * 4 / 0.5)) + 1]
    assert ov.lod_from(per_rad, 3600, 0.0) == [0, 1 << 30, 1 << 30]
    assert ov.lod_from(np.float32(1e-6), 100, 1.0) == [0, 2, 2]
    lv = ov.tile_levels(1000, (np.float32(500.), np.float32(500.)), np.float32(1e-6), 100, 1.0)
    ring = np.maximum(*np.abs(np.mgrid[0:32, 0:32] - 15))
    assert (lv[ring <= 2] == 0).all() and (lv[ring >= 3] == 2).all()


def test_lod_keys_hold_triangles_of_their_tiles_level(tiles_c1):
    """The key rasteriser with levels: every triangle drawn starts on a multiple of its tile's s and lies inside the
    mesh, coarse triangles are drawn, and levels that are all 0 are the reference's mesh"""
    W, H, R = 600, 100, 400
    o = binding.Oracle(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R, viewer_z=2500.)
    vtx, _ = o.vertex_stage(-180.05, 179.95, znear=100., zfar=100000.)
    N = 2 * R
    v = o.viewer()
    eye = (np.float32(v["viewer_cell_i"]), np.float32(v["viewer_cell_j"]))
    per_rad = ov.window(-180.05, 179.95, W, H)[1]
    lv = ov.tile_levels(N, eye, per_rad, W, 2.0)
    assert (lv == 2).any()
    keys = binding.draw_keys(vtx, N, W, H, levels=lv)
    tri = binding.key_triangles(keys, N, lv)
    t = tri[tri != 0xFFFFFFFF].astype(np.int64)
    lod = t >> ov.LOD_SHIFT
    s = 1 << lod
    cell = (t & ov.CELL_MASK) >> 1
    j, i = cell // (N - 1), cell % (N - 1)
    assert (lod == 2).any() and (lod == 0).any()
    assert (j % s == 0).all() and (i % s == 0).all() and (j <= N - 1 - s).all() and (i <= N - 1 - s).all()
    assert (lv[j // ov.TILE_CELLS, i // ov.TILE_CELLS] == lod).all()
    assert np.array_equal(binding.draw_keys(vtx, N, W, H, levels=np.zeros_like(lv)), binding.draw_keys(vtx, N, W, H))
