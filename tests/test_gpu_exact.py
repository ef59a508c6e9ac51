"""Every rendered pixel bit for bit against the unculled exact reference: the renderer's own vertex arithmetic
restated in numpy (oracle/vertex.py, with the device's own angle functions through horizonator_debug_device_math()),
every triangle of the mesh -- or of the level-of-detail set -- drawn without any culling by the oracle's key
rasteriser (glp_draw_keys(), the oracle's rules F2-F8), the minimum key per pixel, and the oracle's read-back.  The
image, the range image and the triangle each pixel shows (horizonator_pick_batch over the whole image, with its cell
number and level bits) must be equal everywhere: culling, the bands, the span grid, the queues and the level of detail
cannot change a pixel.  Run on the B200 box: pytest -m gpu."""
import os
import time

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON
from oracle import binding
from oracle import vertex as ov

pytestmark = pytest.mark.gpu
F = np.float32
SKY = 0xFFFFFFFF
FULL = (-180.05, 179.95)
C2_LAT, C2_LON = 34.0 + 1.0 / 7200.0, -117.0 + 1.0 / 7200.0      # the bench viewpoint (tests/test_gpu_culling.py)
ZEXT = (100., 120000., 100., 120000.)


@pytest.fixture(scope="module")
def hz():
    import horizonator_b200
    return horizonator_b200


def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test running without a CUDA device"
    return torch


class Context:
    """A product context and the exact reference of its views"""

    def __init__(self, hz, tiles, W, H, zext=ZEXT, lod=0.0, seam=False, curvature=False, profiled=False,
                 at=(C1_LAT, C1_LON), **kw):
        self.hz, self.W, self.H, self.zext, self.lod, self.seam = hz, W, H, zext, lod, seam
        self.h = hz.horizonator(at[0], at[1], W, H, dir_dems=tiles, **kw)
        self.h.set_zextents(*zext)
        if lod:
            self.h.set_lod(lod)
        if seam:
            self.h.set_seam_wrap(True)
        if curvature:
            self.h.set_earth_curvature(True)
        if profiled:
            self.h.profile(True)
        self.curv = ov.curvature(curvature)
        self.mosaic = self.h.mosaic()
        self.N = self.mosaic.shape[0]
        d = self.h.context.dems
        self.dem = (d.origin_dem_lon_lat[0], d.origin_dem_lon_lat[1], d.origin_dem_cellij[0], d.origin_dem_cellij[1],
                    d.cells_per_deg)
        self.atan = ov.device_atan(hz.lib)

    def reference(self, view):
        """(image, ranges, triangle) of one view (lat, lon, az0, az1[, viewer_z]), top row first"""
        lat, lon, az0, az1 = view[:4]
        eye = ov.eye(self.dem, self.mosaic, lat, lon, view[4] if len(view) > 4 else -1.0)
        win = ov.window(az0, az1, self.W, self.H, self.seam)
        vtx = ov.grid(self.mosaic, self.N, eye, win, self.W, self.H, self.zext, self.dem[4], self.curv, self.atan)
        levels = ov.tile_levels(self.N, eye, win[1], self.W, self.lod) if self.lod else None
        keys = binding.draw_keys(vtx, self.N, self.W, self.H, win[3], levels)
        img, rng = binding.read_keys(keys, az0, az1, self.zext[0], self.zext[1])
        return img, rng, binding.key_triangles(keys, self.N, levels)

    def pick(self, views):
        """(images, ranges, triangles) of one horizonator_pick_batch_device call over every pixel of the views"""
        torch = _torch()
        n, H, W = len(views), self.H, self.W
        img = torch.full((n, H, W, 3), 0x5A, dtype=torch.uint8, device="cuda")
        rng = torch.full((n, H, W), 7.0, dtype=torch.float32, device="cuda")
        g = torch.full((n, H, W, 32), 0xA5, dtype=torch.uint8, device="cuda")
        self.h.pick_device(views, None, g, d_images=img, d_ranges=rng)
        torch.cuda.synchronize()
        tri = g.cpu().numpy().view(np.dtype(self.hz.GROUND_DTYPE)).reshape(n, H, W)["triangle"]
        return img.cpu().numpy(), rng.cpu().numpy(), tri

    def check(self, views, got=None, what=""):
        """got = (images, ranges[, triangles]) of the views (default: one pick call) against the reference.  A lone view
        must show terrain, and so must most of several (a narrow window can look over all of it)."""
        got = self.pick(views) if got is None else got
        terrain = 0
        for k, v in enumerate(views):
            want = self.reference(v)
            assert_exact(tuple(a[k] for a in got), want, "%s view %d %s" % (what, k, v), need_terrain=len(views) == 1)
            terrain += (want[1] > 0).any()
        assert terrain > 0.6 * len(views), "%s: terrain in %d of %d views: not a test" % (what, terrain, len(views))


def assert_exact(got, want, what, columns=slice(None), need_terrain=True):
    """image, ranges (and triangle) bit for bit; on a difference: which pixels, which triangles"""
    names = ("image", "ranges", "triangle")
    bad = np.zeros(want[1][:, columns].shape, bool)
    for name, a, b in zip(names, got, want):
        a, b = np.ascontiguousarray(a[:, columns]), np.ascontiguousarray(b[:, columns])
        d = a.view(np.uint8).reshape(a.shape[:2] + (-1,)) != b.view(np.uint8).reshape(b.shape[:2] + (-1,))
        bad |= d.any(-1)
    if bad.any():
        ys, xs = np.nonzero(bad)
        rows = []
        for y, x in list(zip(ys, xs))[:12]:
            g = [a[:, columns][y, x] for a in got]
            w = [b[:, columns][y, x] for b in want]
            rows.append("  (y %d, x %d): got %s want %s" % (y, x, _fmt(g), _fmt(w)))
        pytest.fail("%s: %d of %d pixels differ (%d sky / terrain)\n%s" % (
            what, bad.sum(), bad.size, ((want[1][:, columns] == -1) != (got[1][:, columns] == -1)).sum(),
            "\n".join(rows)))
    assert not need_terrain or (want[1][:, columns] > 0).any(), what + ": no terrain in view: not a test"


def _fmt(p):
    s = "img %s range %r" % (tuple(int(c) for c in p[0]), float(p[1]))
    if len(p) > 2:
        t = int(p[2])
        s += " tri sky" if t == SKY else " tri %d (cell %d half %d level %d)" % (t, (t & ov.CELL_MASK) >> 1, t & 1,
                                                                                 t >> ov.LOD_SHIFT)
    return s


def _culled(h):
    c = h.render_counters()
    assert c["tiles_occluded"] > 0 and c["blocks_occluded"] > 0, c
    return c


def _mixed(n, seed, spread=0.4, lat=C1_LAT, lon=C1_LON):
    """n views of different windows (full circle, 90, 5 and 10 degrees, 120, 60) and eye heights"""
    rs = np.random.default_rng(seed)
    v = []
    for k in range(n):
        az0 = float(F(rs.uniform(-180, 180)))
        az1 = float(F(az0 + (360.0, 90.0, 5.0, 120.0, 10.0, 60.0)[k % 6]))
        z = float(F(rs.uniform(1500, 3000))) if k % 4 == 3 else -1.0
        v.append((float(F(lat + rs.uniform(-spread, spread))), float(F(lon + rs.uniform(-spread, spread))), az0, az1, z))
    return v


# ---------------------------------------------------------------------------------------------- scenes (C1 tiles)
SCENES = [
    # name,            W,    H,  R,   az0,     az1,    znear, zfar,   znc,  zfc       (tests/test_gpu_parity.py)
    ("circle_small",   360,  60, 48,  -180.05, 179.95, 100., 100000., -1., -1.),
    ("quarter",        256,  96, 96,   30.0,   120.0,  50.,  20000.,  200., 10000.),
    ("seam_odd_h",     300,  75, 64,   150.0,  210.0,  100., 40000.,  -1., -1.),
    ("narrow_zoom",    400, 100, 200,  80.0,   100.0,  100., 40000.,  -1., -1.),
    ("circle_mid",    1800, 300, 400, -180.05, 179.95, 100., 100000., -1., -1.),
    ("near_clip",      360,  90, 64,  -90.0,   90.0,   5.,   3000.,   -1., -1.),
]


@pytest.mark.parametrize("scene", SCENES, ids=[s[0] for s in SCENES])
def test_scenes(hz, tiles_c1, scene):
    name, W, H, R, az0, az1, zn, zf, znc, zfc = scene
    c = Context(hz, tiles_c1, W, H, (zn, zf, znc if znc > 0 else zn, zfc if zfc > 0 else zf), render_radius_cells=R)
    c.check([(C1_LAT, C1_LON, az0, az1)], what=name)
    # the lone render() of the same view
    img, rng = c.h.render(az0, az1, znear=zn, zfar=zf, znear_color=znc, zfar_color=zfc)
    c.check([(C1_LAT, C1_LON, az0, az1)], got=(img[None], rng[None]), what=name + " render()")


def test_config1_full_size_culls_and_equals_the_reference(hz, tiles_c1):
    c = Context(hz, tiles_c1, 3600, 300, (100., 100000., 100., 100000.), profiled=True, render_radius_cells=1200)
    view = (C1_LAT, C1_LON) + FULL
    c.check([view], got=c.h.render_batch([view]), what="C1 profiled")
    print("C1 counters", _culled(c.h))
    c.h.profile(False)
    c.check([view], what="C1")


def test_eyes_in_a_corner_and_outside_the_square(hz, tiles_c1):
    """A corner eye sees the whole square across the batch bands out to ring 90; an eye beyond the square (explicit
    height) has its tile clamped to the mesh's edge"""
    c = Context(hz, tiles_c1, 1200, 150, profiled=True, render_radius_cells=1200)
    corner = (float(F(C1_LAT - 0.96)), float(F(C1_LON - 0.97))) + FULL
    views = [corner, (float(F(C1_LAT + 1.2)), float(F(C1_LON + 0.3)), -180.05, 179.95, 2200.),
             (float(F(C1_LAT - 1.3)), float(F(C1_LON - 1.1)), 0., 90., 1800.)]
    c.check(views[:1], got=c.h.render_batch(views[:1]), what="corner profiled")
    print("corner counters", _culled(c.h))
    c.check(views, got=c.h.render_batch(views), what="corner/outside profiled")
    c.h.profile(False)
    c.check(views, what="corner/outside")


def test_holes_with_a_moved_viewer(hz, tiles_holes):
    c = Context(hz, tiles_holes, 512, 128, (100., 60000., 100., 60000.), render_radius_cells=500)
    view = (C1_LAT - 0.05, C1_LON + 0.03, -60., 60.)
    c.check([view], what="holes")
    img, rng = c.h.render(-60., 60., lat=view[0], lon=view[1], znear=100., zfar=60000.)
    c.check([view], got=(img[None], rng[None]), what="holes render()")


@pytest.mark.parametrize("R", [1, 2, 3, 17])
def test_tiny_meshes(hz, tiles_c1, R):
    c = Context(hz, tiles_c1, 200, 50, (1., 100000., 1., 100000.), render_radius_cells=R)
    views = [(C1_LAT, C1_LON) + FULL + (float(c.mosaic.min()) + 0.5,), (C1_LAT, C1_LON, -30., 60.)]
    got = c.pick(views)
    for k, v in enumerate(views):
        assert_exact(tuple(a[k] for a in got), c.reference(v), "R=%d view %d" % (R, k), need_terrain=R > 3)


# ---------------------------------------------------------------------------------------------- shapes
@pytest.mark.parametrize("case", [
    # W,    H,   view,                                               zext
    (1234,  77, (C1_LAT, C1_LON) + FULL, ZEXT),
    (300,   75, (C1_LAT, C1_LON, 150., 210.), ZEXT),
    (800,  200, (C1_LAT, C1_LON, 40., 45.), ZEXT),                    # 5 degrees: k_big, middle-sized, 64-bit edges
    (800,  200, (C1_LAT, C1_LON, -100., -90.), ZEXT),                 # 10 degrees
    (1000, 160, (C1_LAT, C1_LON) + FULL + (3000.,), ZEXT),            # an eye 3 km up
    (1000, 160, (C1_LAT, C1_LON) + FULL, (100., 9000., 100., 9000.)),     # far culling
    (1000, 160, (C1_LAT, C1_LON) + FULL, (2500., 120000., 100., 120000.)),  # a large znear
], ids=["1234x77", "300x75", "zoom5", "zoom10", "eye3km", "small_zfar", "large_znear"])
def test_shapes(hz, tiles_c1, case):
    W, H, view, zext = case
    c = Context(hz, tiles_c1, W, H, zext, render_radius_cells=1200)
    c.check([view], what="%dx%d" % (W, H))


# ---------------------------------------------------------------------------------------------- opt-in modes
@pytest.mark.parametrize("mode", [dict(seam=True), dict(curvature=True), dict(lod=0.5), dict(lod=1.0), dict(lod=2.0),
                                  dict(lod=1.0, seam=True)], ids=["seam", "curvature", "lod0.5", "lod1", "lod2",
                                                                  "lod1_seam"])
def test_opt_in_modes(hz, tiles_c1, mode):
    c = Context(hz, tiles_c1, 1200, 200, render_radius_cells=1200, **mode)
    views = [(C1_LAT, C1_LON) + FULL, (C1_LAT, C1_LON) + FULL + (2800.,), (C1_LAT + 0.3, C1_LON - 0.2, 10., 100.)]
    c.check(views, what=str(mode))
    if "lod" in mode:
        tri = c.pick(views[1:2])[2]
        assert ((tri[tri != SKY] >> ov.LOD_SHIFT) > 0).any(), "no coarse band drawn: not a test"


# ---------------------------------------------------------------------------------------------- paths
@pytest.mark.parametrize("n", [1, 7, 64, 65])
def test_batches_of_mixed_views(hz, tiles_c1, n):
    c = Context(hz, tiles_c1, 400, 100, render_radius_cells=600)
    views = _mixed(n, seed=n)
    c.check(views, what="batch of %d" % n)
    if n == 1:
        c.check(views, got=c.h.render_batch(views), what="render_batch of 1")


def test_profiled_batch(hz, tiles_c1):
    c = Context(hz, tiles_c1, 400, 100, profiled=True, render_radius_cells=600)
    views = _mixed(9, seed=3)
    c.check(views, what="profiled")
    assert c.h.profile_read()["renders"] > 0


@pytest.mark.parametrize("x0,x1", [(36, 136), (36, 137), (0, 20)])
def test_wedges(hz, tiles_c1, x0, x1):
    c = Context(hz, tiles_c1, 360, 90, render_radius_cells=400)
    lat, lon = float(F(C1_LAT + 0.1)), float(F(C1_LON - 0.05))
    c.h.pan_zoom(*FULL)
    c.h.move(lat, lon)
    img = np.zeros((90, 360, 3), np.uint8)
    rng = np.zeros((90, 360), np.float32)
    c.h.render_wedge_host(x0, x1, img, rng)
    want = c.reference((lat, lon) + FULL)
    assert_exact((img, rng), want[:2], "wedge [%d, %d)" % (x0, x1), columns=slice(x0, x1))


@pytest.mark.parametrize("env", [{"HORIZONATOR_TRI_CAPACITY": "1000"}, {"HORIZONATOR_BIG_CAPACITY": "50"},
                                 {"HORIZONATOR_BIGTRI_CAPACITY": "7"}], ids=["tri", "big", "record"])
def test_queue_overflows(hz, tiles_c1, env, monkeypatch):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = Context(hz, tiles_c1, 1000, 160, render_radius_cells=420)
    views = [(C1_LAT + 0.02 * k, C1_LON - 0.01 * k) + FULL for k in range(3)] + [(C1_LAT, C1_LON, 40., 45.)]
    c.check(views, what=str(env))
    img, rng = c.h.render(*FULL, znear=ZEXT[0], zfar=ZEXT[1])
    c.check([(C1_LAT, C1_LON) + FULL], got=(img[None], rng[None]), what=str(env) + " render()")


def test_buffer_reuse_across_epochs(hz, tiles_c1):
    """More than twice HZ_KEY_EPOCHS (8) different views one after another through the same view sets, each compared:
    the epoch wraps twice, and span words and keys of earlier renders are left behind each time"""
    c = Context(hz, tiles_c1, 300, 75, render_radius_cells=300)
    rs = np.random.default_rng(17)
    views = [(float(F(C1_LAT + rs.uniform(-0.2, 0.2))), float(F(C1_LON + rs.uniform(-0.2, 0.2))), a0, a1,
              float(F(rs.uniform(1500, 3000))) if k % 3 == 2 else -1.0)
             for k, (a0, a1) in enumerate([FULL, (-20., 70.), (100., 220.)] * 12)]
    for k in range(18):
        c.check(views[2 * k:2 * k + 2], what="pair %d" % k)
        v = views[2 * k]
        img, rng = c.h.render(v[2], v[3], lat=v[0], lon=v[1], znear=ZEXT[0], zfar=ZEXT[1])
        if v[4] < 0:
            c.check([v], got=(img[None], rng[None]), what="render() %d" % k)


# ---------------------------------------------------------------------------------------------- C2
@pytest.fixture(scope="module")
def c2(hz):
    from tools import synth
    tiles = synth.config2_tiles(os.environ.get("HZ_BENCH_TILES", "/tmp/hz_tiles_c2"))
    c = Context(hz, tiles, 3600, 600, (100., 150000., 100., 150000.), profiled=True, at=(C2_LAT, C2_LON),
                SRTM1=True, render_radius_m=150000.)
    return c


@pytest.mark.parametrize("lod", [0.0, 0.5])
def test_config2_bench_viewpoint(c2, lod):
    """BASELINE config 2 at full size: 3600 x 600 over R = 5858 (274 M triangles, all ten bands of a batch)"""
    c2.lod = lod
    c2.h.set_lod(lod)
    try:
        view = (C2_LAT, C2_LON) + FULL
        lone = c2.h.render_batch([view])
        counters = _culled(c2.h)
        t0, p0 = time.time(), time.process_time()
        want = c2.reference(view)
        print("C2 lod %g: reference %.1f s wall, %.1f s CPU; counters %s" % (lod, time.time() - t0,
                                                                            time.process_time() - p0, counters))
        assert_exact((lone[0][0], lone[1][0]), want[:2], "C2 lod %g lone" % lod)
        # two views: a batch view set, with its ten bands
        got = c2.pick([view, view])
        for k in range(2):
            assert_exact(tuple(a[k] for a in got), want, "C2 lod %g batch view %d" % (lod, k))
    finally:
        c2.lod = 0.0
        c2.h.set_lod(0.0)


def test_config2_eye_in_the_corner_tile(c2):
    """An eye in the middle of the mesh's south-west tile (tests/test_gpu_culling.py EYE_TILES): its rings reach the
    far corner, and the mesh's edges clip them on two sides"""
    d = c2.h.context.dems
    ci = cj = ov.TILE_CELLS // 2
    view = (d.origin_dem_lon_lat[1] + (cj + 0.5 + d.origin_dem_cellij[1]) / d.cells_per_deg,
            d.origin_dem_lon_lat[0] + (ci + 0.5 + d.origin_dem_cellij[0]) / d.cells_per_deg) + FULL
    lone = c2.h.render_batch([view])
    _culled(c2.h)
    want = c2.reference(view)
    assert_exact((lone[0][0], lone[1][0]), want[:2], "C2 corner tile lone")
    got = c2.pick([view, view])
    for k in range(2):
        assert_exact(tuple(a[k] for a in got), want, "C2 corner tile batch view %d" % k)
