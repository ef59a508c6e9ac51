"""Ground points of rendered pixels on the GPU (horizonator_pick_batch*, include/horizonator-batch.h): range and sky
against render_batch_device()'s range image of the same renders, the triangle against the rasteriser's own coverage
rule, the ground point against the host restatement (oracle/pick.py), whole-image against query mode, the host call
against the device call, rendering untouched, argument handling, C2 at the bench viewpoint, sharded over NCCL.  Run on
the B200 box: pytest -m gpu."""
import ctypes as C
import math
import os
import socket

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON
from oracle import pick as op

pytestmark = pytest.mark.gpu
SKY = 0xFFFFFFFF


@pytest.fixture(scope="module")
def hz():
    import horizonator_b200
    return horizonator_b200


def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test running without a CUDA device"
    return torch


def _views_c1(n, seed=11):
    """n views: full circle, 90 degrees, 5-degree zooms, 120 and 180 degrees near the square's edge, 60 degrees,
    some with explicit eye heights"""
    rs = np.random.default_rng(seed)
    v = []
    for k in range(n):
        lat, lon = C1_LAT + rs.uniform(-0.25, 0.25), C1_LON + rs.uniform(-0.25, 0.25)
        az0 = rs.uniform(-180, 180)
        kind = k % 6
        az1 = az0 + (360.0, 90.0, 5.0, 120.0, 180.0, 60.0)[kind]
        if kind == 4:
            lat, lon = C1_LAT + 0.93, C1_LON - 0.94 + 0.05 * (k % 24) / 24
        z = float(rs.uniform(1500, 3000)) if k % 4 == 3 else -1.0
        v.append((float(np.float32(lat)), float(np.float32(lon)), float(np.float32(az0)), float(np.float32(az1)), z))
    return v


def _c1(hz, tiles, W, H, mode=None):
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles, render_radius_cells=1200)
    h.set_zextents(100., 120000.)
    if mode == "seam_wrap":
        h.set_seam_wrap(True)
    elif mode == "lod":
        h.set_lod(1.0)
    elif mode == "curvature":
        h.set_earth_curvature(True)
    elif mode == "profiled":
        h.profile(True)
    return h


def _dem(h):
    d = h.context.dems
    return (d.origin_dem_lon_lat[0], d.origin_dem_lon_lat[1], d.origin_dem_cellij[0], d.origin_dem_cellij[1],
            d.cells_per_deg)


def _ranges(h, views):
    torch = _torch()
    rng = torch.empty((len(views), h.height, h.width), dtype=torch.float32, device="cuda")
    h.render_batch_device(views, 0, rng.data_ptr())
    torch.cuda.synchronize()
    return rng.cpu().numpy()


def _device(h, views, pixels=None, stream=0):
    """ground points of one pick_device call: (n, m) for pixels (n, m, 2), else (n, H, W); the output starts poisoned"""
    torch = _torch()
    n = len(views)
    shape = (n, pixels.shape[1]) if pixels is not None else (n, h.height, h.width)
    g = torch.full(shape + (32,), 0xA5, dtype=torch.uint8, device="cuda")
    d_px = torch.as_tensor(np.ascontiguousarray(pixels, np.int32), device="cuda") if pixels is not None else None
    h.pick_device(views, d_px, g, stream=stream)
    torch.cuda.synchronize()
    return g.cpu().numpy().view(np.dtype(_gdt())).reshape(shape)


def _gdt():
    import horizonator_b200
    return horizonator_b200.GROUND_DTYPE


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _check_sky_and_range(g, rng):
    assert np.array_equal(_bits(g["range_m"]), _bits(rng))
    sky = g["triangle"] == SKY
    assert np.array_equal(sky, rng == -1.0)
    for k in ("lat", "lon", "ele_m", "distance_m"):
        assert np.isnan(g[k][sky]).all() and not np.isnan(g[k][~sky]).any(), k


# ---------------------------------------------------------------------------------------------- 1
@pytest.mark.parametrize("mode", [None, "profiled", "seam_wrap", "lod", "curvature"])
def test_range_and_sky_equal_the_range_image(hz, tiles_c1, mode):
    h = _c1(hz, tiles_c1, 400, 100, mode)
    base = _views_c1(24)
    views = [(v[0], v[1], float(np.float32(v[2] + 0.37 * (k // 24))), float(np.float32(v[3] + 0.37 * (k // 24))), v[4])
             for k, v in ((k, base[k % 24]) for k in range(300))]
    for n in (1, 7, 64, 65, 300):
        want = _ranges(h, views[:n])
        g = _device(h, views[:n])
        _check_sky_and_range(g, want)
    assert (g["triangle"] != SKY).mean() > 0.1, mode
    if mode == "lod":
        assert ((g["triangle"][g["triangle"] != SKY] >> 29) > 0).any()      # coarse bands were drawn and read back
    if mode == "profiled":
        assert h.profile_read()["renders"] > 0
        h.profile(False)


# ---------------------------------------------------------------------------------------------- 2
def _snap(a):
    """hz_snap: window coordinate -> 1/256 pixel (oracle rule F2)"""
    t = np.float32(a) * np.float32(256.0)
    if abs(t) < np.float32(8388608.0):
        t = np.floor(t + np.float32(0.5))
    return int(min(max(float(t), -536870912.0), 536870912.0))


def _covers(X, Y, px, py):
    """the rasteriser's edge rule (oracle/gl_pipeline.c F3/F4) on snapped positions for pixel centre (px, py)"""
    Px, Py = px * 256 + 128, py * 256 + 128
    for k in range(3):
        x0, y0, x1, y1 = X[k], Y[k], X[(k + 1) % 3], Y[(k + 1) % 3]
        dx, dy = x1 - x0, y1 - y0
        b = 0 if (dy < 0 or (dy == 0 and dx < 0)) else 1
        if dx * (Py - y0) - dy * (Px - x0) < b:
            return False
    return True


def _sample_terrain(g, count, seed):
    rs = np.random.default_rng(seed)
    k, y, x = np.nonzero(g["triangle"] != SKY)
    pick = rs.choice(len(k), min(count, len(k)), replace=False)
    return k[pick], y[pick], x[pick]


@pytest.mark.parametrize("mode", [None, "seam_wrap", "lod"])
def test_triangle_covers_the_pixel_and_ground_matches_the_oracle(hz, tiles_c1, mode):
    W, H = 600, 150
    h = _c1(hz, tiles_c1, W, H, mode)
    views = _views_c1(12, seed=5)
    g = _device(h, views)
    mosaic = np.pad(h.mosaic(), ((0, 16), (0, 16)))
    N, dem = mosaic.shape[0] - 16, _dem(h)
    atan = op.device_atan(hz.lib)
    ks, ys, xs = _sample_terrain(g, 400, seed=1)
    reproj, coarse = [], 0
    x_, y_, r_ = C.c_double(), C.c_double(), C.c_double()
    for k, y, x in zip(ks, ys, xs):
        v = views[k]
        gp = g[k, y, x]
        tri = int(gp["triangle"])
        eye = op.eye(dem, mosaic, v[0], v[1], v[4])
        win = op.window(v[2], v[3], W, H, seam_wrap=mode == "seam_wrap")
        lat, lon, ele, dist = op.ground(tri, int(x), int(y), mosaic, N, eye, win, W, H, dem, atan=atan)
        # the copy of the triangle the oracle used: its snapped positions cover the pixel centre
        cx = x + 0.5
        covered = False
        for copy in (0, 1, 2):
            xn, xw, yw, vj, vi, z, e, n = op.window_positions(tri, mosaic, N, eye, win, W, H, copy, atan=atan,
                                                              cpd=dem[4])
            if copy > 0 and not (win[3] > 0 and float(xw.min()) <= cx <= float(xw.max())):
                continue
            X, Y = [_snap(a) for a in xw], [_snap(a) for a in yw]
            if _covers(X, Y, int(x), H - 1 - int(y)):
                covered = True
                break
            if copy == 0 and not (win[3] > 0 and float(xn.max() - xn.min()) > 0.5):
                break
        assert covered, (mode, k, y, x, tri)
        lod = tri >> 29
        if lod:
            coarse += 1
            assert all(a % (1 << lod) == 0 for a in vj + vi), (tri, vj, vi)
        assert abs(gp["lat"] - lat) * dem[4] < 1e-6 and abs(gp["lon"] - lon) * dem[4] < 1e-6, (mode, k, y, x)
        assert abs(float(gp["ele_m"]) - ele) < 1e-3 and abs(float(gp["distance_m"]) - dist) <= 1e-6 * dist + 1e-3
        zs = [float(mosaic[a, b]) for a, b in zip(vj, vi)]
        slack = 0.02 * (max(zs) - min(zs)) + 1e-3          # weights up to ~1/256 px outside [0, 1] at silhouettes
        assert min(zs) - slack <= float(gp["ele_m"]) <= max(zs) + slack
        if mode is None:
            cos_lat = math.cos(float(np.float32(v[0])) * math.pi / 180.)
            if hz.lib.horizonator_project(C.byref(x_), C.byref(y_), C.byref(r_), float(np.float32(v[0])), cos_lat,
                                          float(np.float32(v[1])), float(eye[2]), float(gp["lat"]), float(gp["lon"]),
                                          float(gp["ele_m"]), v[2] * math.pi / 180., v[3] * math.pi / 180., W, H):
                reproj.append(math.hypot(x_.value - x, y_.value - y))
    if mode == "lod":
        assert coarse > 0
    if mode is None:
        q = np.percentile(reproj, [50, 90, 99, 100])
        print("\nreprojection of (lat, lon, ele) through horizonator_project(), pixels from the pixel centre, %d pixels: "
              "median %.4f, 90%% %.4f, 99%% %.4f, max %.4f" % (len(reproj), *q))
        assert q[0] < 0.5


# ---------------------------------------------------------------------------------------------- 3
def test_whole_image_equals_query_mode_and_host_equals_device(hz, tiles_c1):
    W, H = 320, 80
    h = _c1(hz, tiles_c1, W, H, "seam_wrap")
    views = _views_c1(70, seed=8)
    whole = _device(h, views)
    yy, xx = np.mgrid[0:H, 0:W]
    allpx = np.stack([xx.ravel(), yy.ravel()], axis=1).astype(np.int32)
    query = _device(h, views, np.broadcast_to(allpx, (len(views),) + allpx.shape))
    assert np.array_equal(query.view(np.uint8).reshape(-1), whole.view(np.uint8).reshape(-1))
    # per-view pixels, some outside the image (sky), on the host
    rs = np.random.default_rng(2)
    px = np.stack([rs.integers(-5, W + 5, (len(views), 500)), rs.integers(-5, H + 5, (len(views), 500))], axis=2)
    px = px.astype(np.int32)
    host = h.pick(views, px)
    dev = _device(h, views, px)
    assert np.array_equal(host.view(np.uint8), dev.view(np.uint8))
    inside = (px[..., 0] >= 0) & (px[..., 0] < W) & (px[..., 1] >= 0) & (px[..., 1] < H)
    assert (host["triangle"][~inside] == SKY).all() and (host["range_m"][~inside] == -1.0).all()
    k = np.nonzero(inside)
    want = whole[k[0], px[..., 1][k], px[..., 0][k]]
    assert np.array_equal(host[k].view(np.uint8), want.view(np.uint8))
    lat, lon, ele, rng = h.ground(views[:5])
    assert np.array_equal(_bits(rng), _bits(whole["range_m"][:5]))
    assert np.array_equal(lat.view(np.uint64), whole["lat"][:5].view(np.uint64))
    # the same pixels for every view
    both = h.pick(views[:3], allpx[:100])
    assert np.array_equal(both.view(np.uint8), whole[:3].reshape(3, -1)[:, :100].view(np.uint8))


# ---------------------------------------------------------------------------------------------- 4
def _legacy_picks(hz, h, W, H):
    """horizonator_pick() over a grid of pixels: (x, y, lat, lon), None where it returns false"""
    lat, lon = C.c_float(), C.c_float()
    out = []
    for x in range(0, W, 37):
        for y in range(0, H, 9):
            ok = hz.lib.horizonator_pick(C.byref(h.context), C.byref(lat), C.byref(lon), x, y)
            out.append((x, y, lat.value, lon.value) if ok else None)
    return out


def test_rendering_untouched_with_picks_interleaved(hz, tiles_c1):
    torch = _torch()
    W, H = 400, 100
    h = _c1(hz, tiles_c1, W, H)
    views = _views_c1(40, seed=3)
    img0 = torch.empty((40, H, W, 3), dtype=torch.uint8, device="cuda")
    rng0 = torch.empty((40, H, W), dtype=torch.float32, device="cuda")
    h.render_batch_device(views, img0.data_ptr(), rng0.data_ptr())
    # lone render (with the same z extents) and the legacy pick
    h.render(views[0][2], views[0][3], lat=views[0][0], lon=views[0][1], znear=100., zfar=120000.)
    legacy = _legacy_picks(hz, h, W, H)
    s = torch.cuda.Stream()
    img1, rng1 = torch.empty_like(img0), torch.empty_like(rng0)
    g = torch.empty((40, H, W, 32), dtype=torch.uint8, device="cuda")
    g2 = torch.empty((40, H, W, 32), dtype=torch.uint8, device="cuda")
    px = torch.zeros((40, 10, 2), dtype=torch.int32, device="cuda")
    gq = torch.empty((40, 10, 32), dtype=torch.uint8, device="cuda")
    with torch.cuda.stream(s):
        h.pick_device(views, None, g, stream=s.cuda_stream)
        h.pick_device(views, px, gq, stream=s.cuda_stream)
        h.render_batch_device(views, img1.data_ptr(), 0, stream=s.cuda_stream)
        h.pick_device(views, None, g2, img1.data_ptr(), rng1.data_ptr(), stream=s.cuda_stream)
    s.synchronize()
    assert torch.equal(img0, img1) and torch.equal(rng0.view(torch.int32), rng1.view(torch.int32))
    assert torch.equal(g, g2)
    gn = g.cpu().numpy().view(_gdt()).reshape(40, H, W)
    _check_sky_and_range(gn, rng0.cpu().numpy())
    h.render(views[0][2], views[0][3], lat=views[0][0], lon=views[0][1], znear=100., zfar=120000.)
    again = _legacy_picks(hz, h, W, H)
    assert again == legacy and any(r is not None for r in legacy)


# ---------------------------------------------------------------------------------------------- 5
def test_invalid_arguments_write_nothing(hz, tiles_c1):
    torch = _torch()
    h = _c1(hz, tiles_c1, 64, 16)
    ctx, lib = C.byref(h.context), hz.lib
    views = h._views([(C1_LAT, C1_LON, 0., 90.)] * 2)
    px = torch.zeros((2, 4, 2), dtype=torch.int32, device="cuda")
    g = torch.full((2, 16, 64, 32), 0xA5, dtype=torch.uint8, device="cuda")
    P, G = px.data_ptr(), g.data_ptr()
    f = lib.horizonator_pick_batch_device
    assert not f(ctx, -1, views, 4, P, G, None, None, None)
    assert not f(ctx, 2, views, -1, P, G, None, None, None)
    assert not f(ctx, 2, None, 4, P, G, None, None, None)
    assert not f(ctx, 2, views, 4, P, None, None, None, None)
    assert not f(ctx, 2, views, 0, None, None, None, None, None)           # whole image without a destination
    assert not f(ctx, 2, views, 4, P + 4, G, None, None, None)             # misaligned pixels
    assert not f(ctx, 2, views, 4, P, G + 4, None, None, None)             # misaligned ground
    assert f(ctx, 0, views, 4, P, G, None, None, None)
    assert f(ctx, 0, None, 0, None, None, None, None, None)
    assert f(ctx, 2, views, 0, P, G, None, None, None)                     # m == 0 with pixels: nothing
    torch.cuda.synchronize()
    assert (g == 0xA5).all().item()
    hp = np.zeros((2, 4, 2), np.int32)
    hg = np.full((2, 4), 0xA5, np.uint8).repeat(32).reshape(2, 4, 32)
    hf = lib.horizonator_pick_batch
    assert not hf(ctx, -1, views, 4, hp.ctypes.data, hg.ctypes.data)
    assert not hf(ctx, 2, views, 4, hp.ctypes.data, None)
    assert not hf(ctx, 2, None, 4, hp.ctypes.data, hg.ctypes.data)
    assert hf(ctx, 2, views, 0, hp.ctypes.data, hg.ctypes.data)
    assert (hg == 0xA5).all()
    assert hf(ctx, 2, views, 4, hp.ctypes.data, hg.ctypes.data) and not (hg == 0xA5).all()
    torch.cuda.synchronize()
    f(ctx, 2, views, 0, None, G, None, None, None)
    torch.cuda.synchronize()
    assert not (g == 0xA5).all().item()


# ---------------------------------------------------------------------------------------------- 6
def test_c2_at_the_bench_viewpoint(hz):
    torch = _torch()
    import bench
    from tools import synth
    C2 = bench.C2
    tiles = synth.config2_tiles(os.environ.get("HZ_BENCH_TILES", "/tmp/hz_tiles_c2"))
    h = hz.horizonator(C2["lat"], C2["lon"], C2["W"], C2["H"], SRTM1=True, dir_dems=tiles, render_radius_m=C2["radius_m"])
    h.set_zextents(C2["znear"], C2["zfar"])
    W, H = C2["W"], C2["H"]
    views = [(C2["lat"], C2["lon"], C2["az0"] + 0.7 * k, C2["az1"] + 0.7 * k) for k in range(256)]
    rng = torch.empty((256, H, W), dtype=torch.float32, device="cuda")
    h.render_batch_device(views, 0, rng.data_ptr())
    rs = np.random.default_rng(9)
    px = np.stack([rs.integers(0, W, (256, 1000)), rs.integers(0, H, (256, 1000))], axis=2).astype(np.int32)
    g = _device(h, views, px)
    want = rng.cpu().numpy()[np.arange(256)[:, None], px[..., 1], px[..., 0]]
    _check_sky_and_range(g, want)
    assert (g["triangle"] != SKY).mean() > 0.01
    whole = torch.empty((256, H, W, 32), dtype=torch.uint8, device="cuda")
    h.pick_device(views, None, whole)
    torch.cuda.synchronize()
    got = whole.view(torch.float32)[..., 5]                    # range_m: bytes 20..23
    assert torch.equal(got.contiguous().view(torch.int32), rng.view(torch.int32))


# ---------------------------------------------------------------------------------------------- 7
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, tiles, q):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    os.environ["HORIZONATOR_DEVICE"] = str(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import horizonator_b200 as hz
        from horizonator_b200 import sharding
        h = hz.horizonator(C1_LAT, C1_LON, 800, 200, dir_dems=tiles, render_radius_cells=600)
        views = [(C1_LAT + 0.011 * k, C1_LON - 0.009 * k, 10. * k, 10. * k + 360.) for k in range(-6, 7)]
        px = np.stack([np.arange(0, 800, 7), np.arange(0, 800, 7) % 200], axis=1)
        want = h.pick(views, px)
        got = sharding.pick_sharded(h, views, px)
        q.put((rank, bool(np.array_equal(got.cpu().numpy().reshape(-1), want.view(np.uint8).reshape(-1)))))
    finally:
        dist.destroy_process_group()


def test_nccl_sharded_picks_equal_one_gpu(tiles_c1):
    import torch
    import torch.multiprocessing as mp
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = min(n, 2)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, tiles_c1, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    got = sorted(q.get(timeout=5) for _ in range(world))
    assert got == [(r, True) for r in range(world)]
