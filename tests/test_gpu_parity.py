"""GPU parity tests proper: the CUDA path, called through the C ABI (ctypes mirror in horizonator_b200),
against the CPU oracle on the same seeded synthetic tiles.  Run on the B200 box: pytest -m gpu.

Bars (BASELINE.json north_star): DEM mosaic bit-exact; coverage agreement >= 99.5 %; range within 1e-4
relative where both hit (exceptions only on silhouette edges, inside the same 0.5 % budget); red +-1 LSB.
Sharded (wedge, batch) renders must equal the unsharded ones bit-for-bit, and repeated renders too.
"""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON
from compare import compare_renders

pytestmark = pytest.mark.gpu


def _torch_cuda():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test running without a CUDA device"
    return torch


@pytest.fixture(scope="module")
def hz():
    import horizonator_b200
    return horizonator_b200


def _oracle(tiles, W, H, R, lat=C1_LAT, lon=C1_LON, **kw):
    from oracle.binding import Oracle
    return Oracle(lat, lon, W, H, SRTM1=False, dir_dems=tiles, render_radius_cells=R, threads=os.cpu_count() or 1, **kw)


# ------------------------------------------------------------------------------------------ K1: mosaic

@pytest.mark.parametrize("R", [1, 5, 48, 600, 1200])
def test_mosaic_bit_exact(hz, tiles_c1, R):
    """k_mosaic vs dem.c:264-309 restated (oracle) for every cell of the square."""
    h = hz.horizonator(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_c1, render_radius_cells=R)
    got = h.mosaic()
    if R <= 48:
        o = _oracle(tiles_c1, 64, 16, R)
        want = o.mosaic()
    else:
        # large squares: assemble the expectation from the raw tiles with numpy (same rule as dem.c)
        want = _numpy_mosaic(tiles_c1, h.context.dems)
    assert got.dtype == np.int16 and got.shape == (2 * R, 2 * R)
    assert np.array_equal(got, want)
    # ... and for every cell against the REFERENCE's own sampler: dem.c compiled unmodified (oracle/_ref), called once
    # per cell in a C loop like horizonator-lib.c:435-439 does
    # (not for R = 1: there the square starts on cell 0 of a tile, where the reference reads out of bounds -- SURVEY Q10,
    # it segfaults -- and the product defines the result instead)
    from oracle import binding
    if binding.have_ref() and R > 1:
        rd = binding.ReferenceDem(C1_LAT, C1_LON, dir_dems=tiles_c1, render_radius_cells=R, threads=os.cpu_count() or 1)
        assert np.array_equal(got, rd.mosaic())
        rd.close()
    # and the host-side sampler of the product agrees with the device copy on a scattered subset
    rs = np.random.default_rng(R)
    for _ in range(200):
        i, j = int(rs.integers(0, 2 * R)), int(rs.integers(0, 2 * R))
        assert hz.lib.horizonator_dem_sample(C.byref(h.context.dems), i, j) == got[j, i]


def _numpy_mosaic(tiles_dir, dems):
    from tools.synth import tile_name
    cpd, R = dems.cells_per_deg, dems.radius_cells
    N = 2 * R
    oi, oj = dems.origin_dem_cellij[0], dems.origin_dem_cellij[1]
    lon0, lat0 = dems.origin_dem_lon_lat[0], dems.origin_dem_lon_lat[1]
    out = np.zeros((N, N), np.int16)
    gi = np.arange(N) + oi
    gj = np.arange(N) + oj

    def split(g):
        t = g // cpd
        c = g - t * cpd
        z = c == 0
        t = np.where(z, t - 1, t)
        c = np.where(z, cpd, c)
        neg = t < 0
        return np.where(neg, 0, t), np.where(neg, 0, c)

    ti, ci = split(gi)
    tj, cj = split(gj)
    cache = {}
    for a in np.unique(ti):
        for b in np.unique(tj):
            path = os.path.join(tiles_dir, tile_name(lat0 + int(b), lon0 + int(a)))
            if os.path.exists(path) and os.path.getsize(path) > 0:
                cache[(a, b)] = np.fromfile(path, dtype=">i2").reshape(cpd + 1, cpd + 1)
            else:
                cache[(a, b)] = None
            cols = np.where(ti == a)[0]
            rows = np.where(tj == b)[0]
            if cache[(a, b)] is None:
                continue
            sub = cache[(a, b)][np.ix_(cpd - cj[rows], ci[cols])]
            out[np.ix_(rows, cols)] = np.maximum(sub, 0)
    return out


def test_mosaic_missing_and_empty_tiles(hz, tiles_holes):
    h = hz.horizonator(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_holes, render_radius_cells=300)
    got = h.mosaic()
    want = _numpy_mosaic(tiles_holes, h.context.dems)
    assert np.array_equal(got, want)
    assert (got[:300, 300:] == 0).all() or (got[300:, :300] == 0).all()   # at least one quadrant is sea


# ------------------------------------------------------------------------------------------ render parity

SCENES = [
    # name,            W,    H,  R,   az0,     az1,    znear, zfar,   znc,  zfc
    ("circle_small",   360,  60, 48,  -180.05, 179.95, 100., 100000., -1., -1.),
    ("quarter",        256,  96, 96,   30.0,   120.0,  50.,  20000.,  200., 10000.),
    ("seam_odd_h",     300,  75, 64,   150.0,  210.0,  100., 40000.,  -1., -1.),
    ("narrow_zoom",    400, 100, 200,  80.0,   100.0,  100., 40000.,  -1., -1.),
    ("circle_mid",    1800, 300, 400, -180.05, 179.95, 100., 100000., -1., -1.),
    ("near_clip",      360,  90, 64,  -90.0,   90.0,   5.,   3000.,   -1., -1.),
]


@pytest.mark.parametrize("scene", SCENES, ids=[s[0] for s in SCENES])
def test_render_matches_oracle(hz, tiles_c1, scene):
    name, W, H, R, az0, az1, znear, zfar, znc, zfc = scene
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    img, rng = h.render(az0, az1, znear=znear, zfar=zfar, znear_color=znc, zfar_color=zfc)
    o = _oracle(tiles_c1, W, H, R)
    img_o, rng_o = o.render(az0, az1, znear=znear, zfar=zfar, znear_color=znc, zfar_color=zfc)
    s = compare_renders(img, rng, img_o, rng_o)
    print(name, s)
    assert s["hit_fraction_ref"] > 0.01, "scene shows no terrain: not a test"
    assert s["ok"], s


def test_config1_full_size(hz, tiles_c1):
    """BASELINE config 1 at full size: R=1200, 3600x300, az [-180.05,179.95], znear 100, zfar 100000."""
    W, H, R = 3600, 300, 1200
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    img, rng = h.render(-180.05, 179.95, znear=100., zfar=100000.)
    o = _oracle(tiles_c1, W, H, R)
    img_o, rng_o = o.render(-180.05, 179.95, znear=100., zfar=100000.)
    s = compare_renders(img, rng, img_o, rng_o)
    print("config1", s, h.last_render_stats())
    assert s["ok"], s


def test_render_moved_viewer_and_holes(hz, tiles_holes):
    W, H, R = 512, 128, 500
    lat, lon = C1_LAT - 0.05, C1_LON + 0.03
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_holes, render_radius_cells=R)
    img, rng = h.render(-60., 60., lat=lat, lon=lon, znear=100., zfar=60000.)
    o = _oracle(tiles_holes, W, H, R)
    img_o, rng_o = o.render(-60., 60., lat=lat, lon=lon, znear=100., zfar=60000.)
    s = compare_renders(img, rng, img_o, rng_o)
    print("moved+holes", s)
    assert s["ok"], s


def test_flat_world_analytic(hz, tmp_path):
    """All tiles missing => elevation 0 everywhere.  Eye 50 m up: ground pixel at elevation el<0 has slant
    range h/sin|el| (linear interpolation inside a cell is exact on a plane through... the eye-centred
    projection is not linear, so allow 1e-3) and the reported range is slant/cos(el) (reference quirk Q1)."""
    W, H, R = 720, 120, 300
    d = d_tiles = str(tmp_path)
    import horizonator_b200 as hb
    ctx = hb.context_t()
    z = C.c_float(50.0)
    assert hb.lib.horizonator_init(C.byref(ctx), C1_LAT, C1_LON, C.byref(z), W, H, R, -1.0, True, False, False,
                                   os.fsencode(d), None, None, None, False)
    try:
        assert hb.lib.horizonator_pan_zoom(C.byref(ctx), -180.05, 179.95)
        assert hb.lib.horizonator_set_zextents(C.byref(ctx), 100., 20000., 100., 20000.)
        img = np.empty((H, W, 3), np.uint8)
        rng = np.empty((H, W), np.float32)
        assert hb.lib.horizonator_render_offscreen(C.byref(ctx), img.ctypes.data, rng.ctypes.data)
    finally:
        hb.lib.horizonator_deinit(C.byref(ctx))
    deg_per_px = 360.0 / W
    rows = np.arange(H)
    el = np.radians((1 - (2 * rows + 1) / H) * (360.0 / (2 * (W / H))))     # SURVEY appendix A
    assert abs(np.degrees(el[0]) - (H / 2 - 0.5) * deg_per_px) < 1e-9
    up = el >= 0
    assert (rng[up] == -1).all() and (img[up] == (255, 0, 0)).all()
    for r in np.where(~up)[0]:
        slant = 50.0 / np.sin(-el[r])
        row = rng[r]
        if 500.0 < slant < 20000.0 * 0.99 and slant * np.cos(el[r]) < 0.8 * R * 92.6 * np.cos(np.radians(35)):
            # columns next to the window seam may be empty: triangles straddling it are dropped, not split
            # (geometry.glsl:15-27; SURVEY appendix B, Q4) -- a gap up to one cell (~93 m) wide
            gap = int(np.ceil(np.degrees(2 * 93.0 / (slant * np.cos(el[r]))) / deg_per_px)) + 1
            assert (row[gap:-gap] > 0).all(), (r, slant)
            # the slant range is interpolated linearly in screen space across a ~93 m cell: seen from distance d
            # the error is of order (cell/d)^2; farther out it converges on the analytic value
            d = slant * np.cos(el[r])
            np.testing.assert_allclose(row[gap:-gap], slant / np.cos(el[r]), rtol=2e-3 + (93.0 / d) ** 2)
        elif slant < 99.0:
            assert (row == -1).all()
    # and the same scene through the oracle (explicit eye height: C API only)
    from oracle.binding import Oracle
    o = Oracle(C1_LAT, C1_LON, W, H, dir_dems=d_tiles, render_radius_cells=R, viewer_z=50.0, threads=os.cpu_count() or 1)
    img_o, rng_o = o.render(-180.05, 179.95, znear=100., zfar=20000.)
    s = compare_renders(img, rng, img_o, rng_o)
    print("flat", s)
    assert s["ok"], s


# ------------------------------------------------------------------------------------------ determinism, shards

def test_repeatable(hz, tiles_c1):
    h = hz.horizonator(C1_LAT, C1_LON, 900, 150, dir_dems=tiles_c1, render_radius_cells=300)
    a = h.render(-180.05, 179.95, zfar=100000.)
    for _ in range(3):
        b = h.render(-180.05, 179.95, zfar=100000.)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_wedges_equal_full_render(hz, tiles_c1):
    torch = _torch_cuda()
    W, H, R = 1200, 200, 300
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    img, rng = h.render(-180.05, 179.95, zfar=100000.)
    for G in (2, 3, 8):
        edges = [W * g // G for g in range(G + 1)]
        out_i = np.empty_like(img)
        out_r = np.empty_like(rng)
        for g in range(G):
            x0, x1 = edges[g], edges[g + 1]
            di = torch.empty((H, x1 - x0, 3), dtype=torch.uint8, device="cuda")
            dr = torch.empty((H, x1 - x0), dtype=torch.float32, device="cuda")
            h.render_wedge_device(x0, x1, di.data_ptr(), dr.data_ptr())
            torch.cuda.synchronize()
            out_i[:, x0:x1] = di.cpu().numpy()
            out_r[:, x0:x1] = dr.cpu().numpy()
        assert np.array_equal(out_i, img), G
        assert np.array_equal(out_r, rng), G


def test_batch_equals_loop(hz, tiles_c1):
    torch = _torch_cuda()
    W, H, R = 600, 100, 200
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    h.set_zextents(100., 50000.)
    views = [(C1_LAT + 0.01 * k, C1_LON - 0.01 * k, -180.05 + 10 * k, 179.95 + 10 * k) for k in range(4)]
    bi, br = h.render_batch(views)
    di = torch.empty((len(views), H, W, 3), dtype=torch.uint8, device="cuda")
    dr = torch.empty((len(views), H, W), dtype=torch.float32, device="cuda")
    h.render_batch_device(views, di.data_ptr(), dr.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(di.cpu().numpy(), bi) and np.array_equal(dr.cpu().numpy(), br)
    for k, (lat, lon, a0, a1) in enumerate(views):
        i1, r1 = h.render(a0, a1, lat=lat, lon=lon, zfar=50000.)
        assert np.array_equal(i1, bi[k]) and np.array_equal(r1, br[k]), k


# ------------------------------------------------------------------------------------------ API behaviour

def test_python_api_shapes_and_errors(hz, tiles_c1):
    h = hz.horizonator(C1_LAT, C1_LON, 128, 32, dir_dems=tiles_c1, render_radius_cells=32)
    assert str(h).startswith("Looking out from 35.00")
    assert h.render(0, 90, return_image=False, return_range=False) == ()
    im = h.render(0, 90, return_range=False)
    assert im.shape == (32, 128, 3) and im.dtype == np.uint8
    r = h.render(0, 90, return_image=False)
    assert r.shape == (32, 128) and r.dtype == np.float32
    a = h.render(0, 90)
    b = h.render(0 + 45. / 127, 90 - 45. / 127 * 0, az_extents_use_pixel_centers=False)
    assert isinstance(a, tuple) and len(a) == 2 and isinstance(b, tuple)
    with pytest.raises(RuntimeError):
        h.render(0, 90, znear=-5.)                        # set_zextents refuses non-positive values
    with pytest.raises(RuntimeError):
        hz.horizonator(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_c1, render_radius_cells=10, render_radius_m=5000.)
    with pytest.raises(RuntimeError):
        hz.horizonator(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_c1, render_texture=True, render_radius_cells=10)
    # pixel-centre convention widens the window by half a pixel each side (pywrap.c:204-212)
    c = h.render(0., 90., az_extents_use_pixel_centers=True)
    half = 90. / 127 / 2
    d = h.render(0. - half, 90. + half)
    assert np.array_equal(c[0], d[0]) and np.array_equal(c[1], d[1])


def test_pick_matches_reference_formula(hz, tiles_c1):
    W, H, R = 360, 60, 64
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    img, rng = h.render(-180.05, 179.95, zfar=100000.)
    ys, xs = np.where(rng > 0)
    assert len(ys) > 10
    lat, lon = C.c_float(), C.c_float()
    for k in range(0, len(ys), max(1, len(ys) // 25)):
        x, y = int(xs[k]), int(ys[k])
        assert hz.lib.horizonator_pick(C.byref(h.context), C.byref(lat), C.byref(lon), x, y)
        # the picked point lies within the loaded square, in the direction of the pixel's azimuth
        az = np.radians(-180.05 + (x + 0.5) / W * 360.0)
        de = (lon.value - C1_LON) * np.cos(np.radians(C1_LAT))
        dn = lat.value - C1_LAT
        assert abs(np.arctan2(de, dn) - az + 2 * np.pi * np.round((az - np.arctan2(de, dn)) / (2 * np.pi))) < 0.05
    ys, xs = np.where(rng < 0)
    assert not hz.lib.horizonator_pick(C.byref(h.context), C.byref(lat), C.byref(lon), int(xs[0]), int(ys[0]))


def test_windowed_context_redraw_and_resize(hz, tiles_c1):
    import horizonator_b200 as hb
    ctx = hb.context_t()
    assert hb.lib.horizonator_init(C.byref(ctx), C1_LAT, C1_LON, None, 0, 0, 32, -1.0, False, False, False,
                                   os.fsencode(tiles_c1), None, None, None, False)
    try:
        assert not ctx.offscreen.inited and ctx.Ntriangles == 2 * 63 * 63
        assert hb.lib.horizonator_redraw(C.byref(ctx))
        assert hb.lib.horizonator_resized(C.byref(ctx), 640, 200)
        assert hb.lib.horizonator_redraw(C.byref(ctx))
        assert not hb.lib.horizonator_render_offscreen(C.byref(ctx), None, None)
    finally:
        hb.lib.horizonator_deinit(C.byref(ctx))
        hb.lib.horizonator_deinit(C.byref(ctx))      # idempotent


def test_reference_python_binding_on_this_library(hz, tiles_c1):
    """Drop-in proof: the reference's own horizonator-pywrap.c, compiled unmodified against include/ and linked
    to libhorizonator.so (oracle/Makefile target `pywrap`), drives the CUDA renderer and returns exactly what
    the ctypes mirror returns."""
    import importlib.util
    import glob
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    so = glob.glob(os.path.join(root, "oracle", "_ref", "pywrap", "horizonator*.so"))
    if not so:
        pytest.skip("oracle/_ref/pywrap was not built (needs /root/reference at build time)")
    spec = importlib.util.spec_from_file_location("horizonator", so[0])
    ref_binding = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_binding)
    W, H, R = 360, 60, 100
    a = ref_binding.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    b = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    assert str(a) == str(b)
    for kw in (dict(), dict(az_extents_use_pixel_centers=True, zfar=80000.),
               dict(lat=C1_LAT + 0.01, lon=C1_LON + 0.01, znear=50., zfar=30000., znear_color=500., zfar_color=20000.)):
        ia, ra = a.render(-100., 80., **kw)
        ib, rb = b.render(-100., 80., **kw)
        assert ia.dtype == ib.dtype and ra.dtype == rb.dtype and ia.shape == ib.shape
        assert np.array_equal(ia, ib) and np.array_equal(ra, rb)
    assert a.render(0., 90., return_image=False, return_range=False) == ()
    assert a.render(0., 90., return_range=False).shape == (H, W, 3)


# ------------------------------------------------------------------------------------------ rarely taken paths

@pytest.mark.parametrize("env,profiled", [
    ({"HORIZONATOR_TRI_CAPACITY": "1000"}, False),                        # triangle list overflows: drawn in the mesh kernel
    ({"HORIZONATOR_BIG_CAPACITY": "50"}, False),                          # sub-box queue overflows
    ({"HORIZONATOR_BIGTRI_CAPACITY": "7"}, False),                        # record pool overflows
    ({}, True),                                                           # the eager chain, k_big of the near pass in line
], ids=["tri_overflow", "big_overflow", "record_overflow", "profiled"])
def test_overflow_paths_and_profiling_do_not_change_the_image(hz, tiles_c1, env, profiled, monkeypatch):
    """Queue overflows fall back to a slow in-kernel path, and a profiled render launches the kernels one by one
    instead of replaying a captured graph: the image must be the one the default configuration produces, bit for bit."""
    W, H, R = 1000, 160, 420
    h0 = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    want = h0.render(-180.05, 179.95, zfar=100000.)
    del h0
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    h1 = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    if profiled:
        h1.profile(True)
    got = h1.render(-180.05, 179.95, zfar=100000.)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    views = [(C1_LAT + 0.02 * k, C1_LON - 0.01 * k, -180.05, 179.95) for k in range(3)]
    h1.set_zextents(100., 100000.)
    bi, br = h1.render_batch(views)
    if profiled:
        assert h1.profile_read()["renders"] == 2        # the single render and the batch's one chunk
    for k, (la, lo, a0, a1) in enumerate(views):
        for key in env:
            monkeypatch.delenv(key)
        hk = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
        wi, wr = hk.render(a0, a1, lat=la, lon=lo, zfar=100000.)
        for key, v in env.items():
            monkeypatch.setenv(key, v)
        assert np.array_equal(bi[k], wi) and np.array_equal(br[k], wr), k


def test_batch_with_more_windows_than_table_slots(hz, tiles_c1):
    """Many distinct azimuth spans in one batch (each needs its own per-row tangent table; round 1 kept 8 in a shared
    cache that a batch could overrun): the batch still equals the loop of single renders."""
    W, H, R = 400, 80, 150
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    h.set_zextents(100., 50000.)
    views = [(C1_LAT, C1_LON, -30.0 - k, 30.0 + 2 * k) for k in range(35)]
    bi, br = h.render_batch(views)
    for k, (la, lo, a0, a1) in enumerate(views):
        wi, wr = h.render(a0, a1, lat=la, lon=lo, zfar=50000.)
        assert np.array_equal(bi[k], wi) and np.array_equal(br[k], wr), k


# chunks of up to 64 views on up to 4 view sets (render_batch_common): 1 view is rendered on the context's own scratch;
# 5 views are one chunk; 37 are chunks of 10/10/10/7 on four sets, the last one ragged; 257 are four chunks of 64, then
# set 0 again, while in flight, for 1 view
@pytest.mark.parametrize("n", [1, 5, 37, 257])
def test_ragged_mixed_batch_equals_single_renders(hz, tiles_c1, n):
    """A batch is rendered in chunks by launches with a view dimension: more views than one chunk holds, a ragged last
    chunk, wide and zoomed-in windows (different chain shapes) and explicit eye heights in one call -- every view must
    equal its single render bit for bit, whatever the chunking."""
    torch = _torch_cuda()
    W, H, R = 480, 96, 180
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    h.set_zextents(100., 60000.)
    rs = np.random.RandomState(5)
    views = []
    for k in range(n):
        la, lo = C1_LAT + rs.uniform(-0.05, 0.05), C1_LON + rs.uniform(-0.05, 0.05)
        c = rs.uniform(-180, 180)
        half = (180.0, 45.0, 6.0)[k % 3]
        z = -1.0 if k % 4 else float(rs.uniform(800, 3000))
        views.append((la, lo, c - half, c + half - (0.1 if half == 180.0 else 0.0), z))
    di = torch.empty((len(views), H, W, 3), dtype=torch.uint8, device="cuda")
    dr = torch.empty((len(views), H, W), dtype=torch.float32, device="cuda")
    d2 = torch.empty_like(di)
    r2 = torch.empty_like(dr)
    stream = torch.cuda.Stream()        # a real stream: the calls only enqueue (stream 0 = NULL would make them synchronous)
    for rep in range(2):        # the second pass replays the captured graphs
        di.zero_(); dr.zero_(); d2.zero_(); r2.zero_()
        torch.cuda.synchronize()
        # two calls back to back without waiting: the second reuses the view sets while the first is still in flight
        h.render_batch_device(views, di.data_ptr(), dr.data_ptr(), stream.cuda_stream)
        h.render_batch_device(views[::-1], d2.data_ptr(), r2.data_ptr(), stream.cuda_stream)
        torch.cuda.synchronize()
        assert torch.equal(d2.flip(0), di) and torch.equal(r2.flip(0), dr)
        bi, br = di.cpu().numpy(), dr.cpu().numpy()
        hi, hr = h.render_batch(views)
        assert np.array_equal(hi, bi) and np.array_equal(hr, br)
        for k, (la, lo, a0, a1, z) in enumerate(views):
            h.move(la, lo, viewer_z=None if z < 0 else z)
            h.pan_zoom(a0, a1)
            wi = hz.pinned_array((H, W, 3), np.uint8); wr = hz.pinned_array((H, W), np.float32)
            h.render_into(wi, wr)
            assert np.array_equal(bi[k], wi) and np.array_equal(br[k], wr), (rep, k)
    # image only / ranges only
    h.render_batch_device(views[:7], di.data_ptr(), 0, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(di[:7].cpu().numpy(), bi[:7])
    dr.zero_()
    h.render_batch_device(views[:7], 0, dr.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(dr[:7].cpu().numpy(), br[:7])


# ------------------------------------------------------------------------------------------ opt-in accuracy mode

def test_earth_curvature_is_opt_in_and_matches_the_extended_oracle(hz, tiles_c1):
    """Off by default (flat earth like the reference).  On: every vertex drops by (1-k) d^2 / (2 R_earth), in the
    CUDA path and in the oracle's opt-in extension alike; far terrain sinks, near terrain stays."""
    W, H, R = 1800, 300, 600
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    flat_i, flat_r = h.render(-180.05, 179.95, zfar=100000.)
    h.set_earth_curvature(True, 0.13)
    img, rng = h.render(-180.05, 179.95, zfar=100000.)
    o = _oracle(tiles_c1, W, H, R)
    o.set_curvature(np.float32((1.0 - np.float32(0.13)) / np.float32(2.0 * 6371000.0)))
    img_o, rng_o = o.render(-180.05, 179.95, zfar=100000.)
    s = compare_renders(img, rng, img_o, rng_o)
    print("curved", s)
    assert s["ok"], s
    assert not np.array_equal(rng, flat_r)
    # the skyline of far terrain is lower (larger row index) with curvature, never higher by more than a pixel
    def skyline(r):
        hit = r > 0
        top = np.where(hit.any(axis=0), hit.argmax(axis=0), -1)
        return top, np.where(top >= 0, r[np.clip(top, 0, H - 1), np.arange(W)], -1.0)
    t_flat, d_flat = skyline(flat_r)
    t_curv, _ = skyline(rng)
    far = (d_flat > 30000.) & (t_curv >= 0)
    assert far.sum() > 50
    assert (t_curv[far] >= t_flat[far] - 1).all() and (t_curv[far] > t_flat[far]).mean() > 0.3
    # and switching it off restores the reference behaviour bit for bit
    h.set_earth_curvature(False)
    again_i, again_r = h.render(-180.05, 179.95, zfar=100000.)
    assert np.array_equal(again_i, flat_i) and np.array_equal(again_r, flat_r)
    with pytest.raises(RuntimeError):
        h.set_earth_curvature(True, 1.5)


def test_renders_on_different_streams_do_not_trample_each_other(hz, tiles_c1):
    """The context's scratch set is shared by the single-view entry points whatever stream they are given: a render
    queued on one stream right after one on another must wait for it (GPU-side), not corrupt it."""
    torch = _torch_cuda()
    W, H, R = 1200, 200, 500
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    h.set_zextents(100., 100000.)
    va = [(C1_LAT, C1_LON, -180.05, 179.95)]
    vb = [(C1_LAT + 0.05, C1_LON - 0.04, -180.05, 179.95)]
    want_a = h.render(-180.05, 179.95, lat=va[0][0], lon=va[0][1], zfar=100000.)
    want_b = h.render(-180.05, 179.95, lat=vb[0][0], lon=vb[0][1], zfar=100000.)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    ia = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda"); ra = torch.empty((H, W), dtype=torch.float32, device="cuda")
    ib = torch.empty_like(ia); rb = torch.empty_like(ra)
    for _ in range(10):
        h.render_batch_device(va, ia.data_ptr(), ra.data_ptr(), s1.cuda_stream)
        h.render_batch_device(vb, ib.data_ptr(), rb.data_ptr(), s2.cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(ia.cpu().numpy(), want_a[0]) and np.array_equal(ra.cpu().numpy(), want_a[1])
    assert np.array_equal(ib.cpu().numpy(), want_b[0]) and np.array_equal(rb.cpu().numpy(), want_b[1])


def test_seam_wrap_is_opt_in_and_closes_the_full_circle(hz, tiles_c1):
    """Off by default: triangles across the +-180 degree seam are dropped like the reference does (geometry.glsl:15-27),
    leaving gaps in the edge columns.  On: they are drawn at both edges, in the CUDA path and in the oracle's opt-in
    extension alike; everything away from the edges is unchanged."""
    W, H, R = 1440, 240, 300
    az0, az1 = -180.0, 179.99                       # seam looking due south; 359.99 degrees wide
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    base_i, base_r = h.render(az0, az1, zfar=60000.)
    h.set_seam_wrap(True)
    img, rng = h.render(az0, az1, zfar=60000.)
    o = _oracle(tiles_c1, W, H, R)
    o.set_seam_wrap(True)
    img_o, rng_o = o.render(az0, az1, zfar=60000.)
    s = compare_renders(img, rng, img_o, rng_o)
    print("wrapped", s)
    assert s["ok"], s
    # a seam triangle is at most a quarter of the window wide (wider ones stay dropped), so beyond that distance from
    # the edges nothing changes; at the edges terrain is gained and none is lost
    m = W // 4 + 2
    assert np.array_equal(rng[:, m:-m], base_r[:, m:-m]) and np.array_equal(img[:, m:-m], base_i[:, m:-m])
    edge = np.r_[0:3, W - 3:W]
    gained = (rng[:, edge] > 0).sum() - (base_r[:, edge] > 0).sum()
    assert gained > 0, gained
    assert ((base_r[:, edge] > 0) <= (rng[:, edge] > 0)).all()
    # in the wrapped render the first and the last column see (nearly) the same terrain rows: the circle closes
    top = lambda col: int(np.argmax(rng[:, col] > 0))
    assert abs(top(0) - top(W - 1)) <= 2
    h.set_seam_wrap(False)
    again_i, again_r = h.render(az0, az1, zfar=60000.)
    assert np.array_equal(again_i, base_i) and np.array_equal(again_r, base_r)


@pytest.mark.parametrize("R,W,H", [(1, 64, 32), (2, 90, 45), (3, 128, 48), (17, 200, 60)])
def test_tiny_meshes(hz, tiles_c1, R, W, H):
    """Meshes smaller than one culling block / tile, down to the single cell of R=1."""
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    img, rng = h.render(-180.05, 179.95, znear=1., zfar=10000.)
    o = _oracle(tiles_c1, W, H, R)
    img_o, rng_o = o.render(-180.05, 179.95, znear=1., zfar=10000.)
    assert np.array_equal(h.mosaic(), o.mosaic())
    s = compare_renders(img, rng, img_o, rng_o)
    print("tiny", R, s)
    assert s["ok"], s


def test_eye_outside_the_loaded_square(hz, tiles_c1):
    """horizonator_move() does not reload DEMs (horizonator.h:120-122): the eye may leave the square, and then sees it
    from outside (every mesh rectangle in one quadrant, the eye's tile clamped to the edge)."""
    W, H, R = 600, 120, 200
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    o = _oracle(tiles_c1, W, H, R)
    for dlat, dlon in ((0.3, 0.25), (-0.21, 0.0), (0.0, -0.4)):
        kw = dict(lat=C1_LAT + dlat, lon=C1_LON + dlon, znear=100., zfar=100000.)
        img, rng = h.render(-180.05, 179.95, **kw)
        img_o, rng_o = o.render(-180.05, 179.95, **kw)
        s = compare_renders(img, rng, img_o, rng_o)
        print("outside", dlat, dlon, s)
        assert s["hit_fraction_ref"] > 0.0005
        assert s["ok"], s


def test_random_views_match_oracle(hz, tiles_c1):
    """Differential test over random eye positions, azimuth windows (5..360 degrees, any orientation), depth extents,
    image shapes and mesh sizes: the conservative culling (quadrant logic, window seam, far/near clip, occlusion)
    must never show in the image."""
    rs = np.random.default_rng(20260117)
    worst = 1.0
    for case in range(36):
        R = int(rs.choice([40, 90, 150, 260]))
        W = int(rs.integers(16, 200)) * 4
        H = int(rs.integers(24, 160))
        half = R / 1200.0 * 0.8
        lat = C1_LAT + float(rs.uniform(-half, half))
        lon = C1_LON + float(rs.uniform(-half, half))
        span = float(rs.choice([5., 17., 45., 90., 180., 270., 359.9]))
        az0 = float(rs.uniform(-360., 360.))
        znear = float(rs.choice([1., 30., 100., 400.]))
        zfar = float(rs.choice([3000., 12000., 40000., 100000.]))
        znc, zfc = (-1., -1.) if rs.uniform() < 0.5 else (float(rs.uniform(10., 500.)), float(rs.uniform(2000., 30000.)))
        h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
        o = _oracle(tiles_c1, W, H, R)
        kw = dict(lat=lat, lon=lon, znear=znear, zfar=zfar, znear_color=znc, zfar_color=zfc)
        img, rng = h.render(az0, az0 + span, **kw)
        img_o, rng_o = o.render(az0, az0 + span, **kw)
        s = compare_renders(img, rng, img_o, rng_o)
        worst = min(worst, s["agreement"])
        assert s["ok"], (case, R, W, H, lat, lon, az0, span, znear, zfar, s)
    print("random views: worst agreement", worst)


def _golden_scenes():
    g = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    return sorted(f[len("render_"):-len(".npz")] for f in os.listdir(g) if f.startswith("render_"))


@pytest.mark.parametrize("name", _golden_scenes())
def test_render_matches_committed_golden_vectors(hz, tiles_c1, name):
    """The CUDA path against the fixtures of tests/golden/ directly: renders recorded from the reference's own
    horizonator-lib.c + dem.c (compiled unmodified; tests/golden/make_golden.py) -- no oracle library involved."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "render_%s.npz" % name))
    W, H, R, az0, az1, zn, zf, znc, zfc, lat, lon = g["params"]
    h = hz.horizonator(C1_LAT, C1_LON, int(W), int(H), dir_dems=tiles_c1, render_radius_cells=int(R))
    kw = {} if lat <= -1000. else dict(lat=float(lat), lon=float(lon))
    img, rng = h.render(float(az0), float(az1), znear=float(zn), zfar=float(zf), znear_color=float(znc),
                        zfar_color=float(zfc), **kw)
    s = compare_renders(img, rng, g["image"], g["ranges"])
    print("golden", name, s)
    assert s["ok"], s


# ------------------------------------------------------------------------------------------ a real GL driver

def _llvmpipe_scenes():
    g = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    return sorted(f[len("llvmpipe_"):-len(".npz")] for f in os.listdir(g) if f.startswith("llvmpipe_") and f.endswith(".npz"))


def _render_c_api(hb, tiles, W, H, R, az0, az1, zn, zf, znc, zfc, lat, lon, vz):
    """One render through the C ABI with an explicit eye height (the Python API has none, like the reference's)."""
    ctx = hb.context_t()
    z = C.c_float(vz)
    assert hb.lib.horizonator_init(C.byref(ctx), C1_LAT, C1_LON, C.byref(z), W, H, R, -1.0, True, False, False,
                                   os.fsencode(tiles), None, None, None, False)
    try:
        assert hb.lib.horizonator_pan_zoom(C.byref(ctx), az0, az1)
        if lat > -1000.:
            assert hb.lib.horizonator_move(C.byref(ctx), None, lat, lon)
        assert hb.lib.horizonator_set_zextents(C.byref(ctx), zn, zf, znc, zfc)
        img = np.empty((H, W, 3), np.uint8)
        rng = np.empty((H, W), np.float32)
        assert hb.lib.horizonator_render_offscreen(C.byref(ctx), img.ctypes.data, rng.ctypes.data)
    finally:
        hb.lib.horizonator_deinit(C.byref(ctx))
    return img, rng


@pytest.mark.parametrize("name", _llvmpipe_scenes())
def test_render_matches_reference_on_llvmpipe(hz, tiles_c1, name):
    """The CUDA path against renders of the UNMODIFIED reference on a real OpenGL implementation (Mesa llvmpipe;
    tests/golden/make_golden_llvmpipe.py) -- neither the oracle nor its GL restatement is involved."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "llvmpipe_%s.npz" % name))
    W, H, R, az0, az1, zn, zf, znc, zfc, lat, lon, vz = (float(x) for x in g["params"])
    img, rng = _render_c_api(hz, tiles_c1, int(W), int(H), int(R), az0, az1, zn, zf, znc, zfc, lat, lon, vz)
    s = compare_renders(img, rng, g["image"], g["ranges"])
    print("llvmpipe", name, s)
    assert s["ok"], s
    assert s["coverage_agreement"] >= 0.9995, s
