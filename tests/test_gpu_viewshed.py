"""Viewsheds on the GPU (horizonator_viewshed*, include/horizonator-batch.h) against the CPU oracle's restatement of
the same definition, bit for bit; batches against lone views; counts against the masks; argument handling; agreement
with what the renderer draws; sharded counts over NCCL.  Run on the B200 box: pytest -m gpu."""
import ctypes as C
import os
import socket

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON
from oracle.viewshed import ViewshedOracle, unpack_mask

pytestmark = pytest.mark.gpu

CURVATURE = np.float32((1.0 - np.float32(0.13)) / np.float32(2.0 * 6371000.0))   # set_earth_curvature(True, 0.13)
C1_EYES = [(C1_LAT, C1_LON), (C1_LAT + 0.03, C1_LON - 0.02), (C1_LAT - 0.04, C1_LON + 0.05)]


@pytest.fixture(scope="module")
def hz():
    import horizonator_b200
    return horizonator_b200


def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test running without a CUDA device"
    return torch


def _oracle(tiles, R, srtm1=False, lat=C1_LAT, lon=C1_LON):
    from oracle.binding import Oracle
    return Oracle(lat, lon, 64, 16, SRTM1=srtm1, dir_dems=tiles, render_radius_cells=R, threads=os.cpu_count() or 1)


def _words_device(h, views, target_height=0.):
    torch = _torch()
    N = h.size
    d = torch.empty((len(views), N, (N + 31) // 32), dtype=torch.int32, device="cuda")
    h.viewshed_device(views, d_masks=d.data_ptr(), target_height=target_height)
    return d.cpu().numpy().view(np.uint32)


@pytest.mark.parametrize("curved", [False, True])
def test_c1_masks_bit_identical_to_the_oracle(hz, tiles_c1, curved):
    R = 1200
    h = hz.horizonator(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_c1, render_radius_cells=R)
    o = _oracle(tiles_c1, R)
    vs = ViewshedOracle(o)
    curvature = CURVATURE if curved else 0.
    if curved:
        h.set_earth_curvature(True, 0.13)
    for th in (0.0, 1.7):
        got = _words_device(h, C1_EYES, th)
        for k, (lat, lon) in enumerate(C1_EYES):
            o.move(lat, lon)
            want = vs.words(th, curvature=curvature)
            assert np.array_equal(got[k], want), (k, th, curved, int((got[k] != want).sum()))
            assert 0.001 < unpack_mask(want).mean() < 0.9
    # the host-memory call returns the same, unpacked
    m = h.viewshed(C1_EYES, 1.7)
    o.move(*C1_EYES[1])
    assert m.shape == (3, 2 * R, 2 * R) and np.array_equal(m[1], vs.mask(1.7, curvature=curvature))


def test_c2_mask_bit_identical_to_the_oracle_at_the_bench_viewpoint(hz):
    from tools import synth
    tiles = synth.config2_tiles(os.environ.get("HZ_BENCH_TILES", "/tmp/hz_tiles_c2"))
    lat, lon = 34.0 + 1.0 / 7200.0, -117.0 + 1.0 / 7200.0
    h = hz.horizonator(lat, lon, 64, 16, SRTM1=True, dir_dems=tiles, render_radius_m=150000.)
    assert h.size == 11716
    got = _words_device(h, [(lat, lon)])[0]
    h.close()
    from oracle.binding import Oracle
    o = Oracle(lat, lon, 64, 16, SRTM1=True, dir_dems=tiles, render_radius_m=150000., threads=os.cpu_count() or 1)
    want = ViewshedOracle(o).words()
    print("C2 visible fraction", float(np.unpackbits(want.view(np.uint8)).mean()))
    assert np.array_equal(got, want), int((got != want).sum())


def test_batch_equals_lone_views_across_chunks(hz, tiles_c1):
    """100 views = two launches of up to 64: view k of the batch is view k run alone; unused bits stay 0."""
    h = hz.horizonator(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_c1, render_radius_cells=400)
    rs = np.random.default_rng(3)
    views = [(C1_LAT + rs.uniform(-0.3, 0.3), C1_LON + rs.uniform(-0.3, 0.3), 0., 0., -1. if k % 3 else 40.)
             for k in range(100)]
    batch = _words_device(h, views, 1.7)
    N = h.size
    tail = np.uint32((1 << (N % 32)) - 1) if N % 32 else np.uint32(0xFFFFFFFF)
    assert not (batch[:, :, -1] & ~tail).any()
    for k, v in enumerate(views):
        assert np.array_equal(_words_device(h, [v], 1.7)[0], batch[k]), k


def test_counts_are_the_sum_of_the_masks_and_accumulate(hz, tiles_c1):
    torch = _torch()
    h = hz.horizonator(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_c1, render_radius_cells=300)
    N = h.size
    views = [(C1_LAT + 0.01 * k, C1_LON - 0.007 * k) for k in range(-4, 5)]
    masks = torch.empty((len(views), N, (N + 31) // 32), dtype=torch.int32, device="cuda")
    counts = torch.zeros((N, N), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()                        # the context's own stream does not wait for torch's fill
    h.viewshed_device(views, d_masks=masks.data_ptr(), d_counts=counts.data_ptr())
    m = unpack_mask(masks.cpu().numpy().view(np.uint32))
    want = m.sum(axis=0)
    assert np.array_equal(counts.cpu().numpy(), want) and want.max() > 1
    h.viewshed_device(views, d_counts=counts.data_ptr())                 # counts only: the scratch path
    assert np.array_equal(counts.cpu().numpy(), 2 * want)
    hm, hc = h.viewshed(views, counts=True)                              # host memory
    assert np.array_equal(hm, m) and np.array_equal(hc, want)


def test_degenerate_and_invalid_arguments_write_nothing(hz, tiles_c1):
    torch = _torch()
    h = hz.horizonator(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_c1, render_radius_cells=200)
    N = h.size
    ctx = C.byref(h.context)
    masks = torch.full((2, N, (N + 31) // 32), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    counts = torch.full((N, N), 7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    lib = hz.lib
    ok = [(C1_LAT, C1_LON)]
    assert lib.horizonator_viewshed_device(ctx, 0, h._eyes(ok), 0., masks.data_ptr(), counts.data_ptr(), None)
    assert not lib.horizonator_viewshed_device(ctx, 1, h._eyes(ok), 0., None, None, None)
    outside = [(C1_LAT, C1_LON), (C1_LAT + 0.2, C1_LON)]                 # R = 200 cells = 0.167 degrees
    assert not lib.horizonator_viewshed_device(ctx, 2, h._eyes(outside), 0., masks.data_ptr(), counts.data_ptr(), None)
    torch.cuda.synchronize()
    assert (masks == 0x5A5A5A5A).all().item() and (counts == 7).all().item()
    hm = np.full((2, N, (N + 31) // 32), 0x5A5A5A5A, np.uint32)
    hc = np.full((N, N), 7, np.uint32)
    assert lib.horizonator_viewshed(ctx, 0, h._eyes(ok), 0., hm.ctypes.data, hc.ctypes.data)
    assert not lib.horizonator_viewshed(ctx, 1, h._eyes(ok), 0., None, None)
    assert not lib.horizonator_viewshed(ctx, 2, h._eyes(outside), 0., hm.ctypes.data, hc.ctypes.data)
    assert (hm == 0x5A5A5A5A).all() and (hc == 7).all()
    with pytest.raises(RuntimeError):
        h.viewshed(outside)


def test_consistent_with_the_renderer(hz, tiles_c1):
    """Vertices 1-5 km from the eye (a cell there spans several pixels at 0.1 degree per pixel), each projected to its
    pixel of a full-circle render (znear 1 m, zfar beyond the square).  The range image holds the slant range over
    cos(elevation of the row) (quirk Q1), so the ratio of a pixel's range to the vertex's own range converted the same
    way is the ratio of slant ranges.  A hidden vertex should have nearer terrain (ratio < 0.98) in its pixel, a
    visible one should not.

    A pixel centre is up to half a pixel from the vertex: within a pixel of a silhouette it may see past the crest that
    hides the vertex, or catch the crest in front of a visible one.  Only vertices whose 3x3 pixel neighbourhood is
    unanimous (all nearer, or none) decide.  Measured at C1, eye (C1 + 0.03, C1 - 0.02 degrees), 10 731 vertices in the
    ring, 83 % decidable: hidden with nearer terrain 0.943, visible without 0.938.  With brute-force line of sight in
    place of R2 (vs_oracle_exact) the figures are 0.943 / 1.000: the visible side's shortfall is R2's
    approximation (169 of its 940 visible vertices in the ring are hidden to exact line of sight), the hidden side's is
    the criterion (a vertex hidden by its own neighbouring cells on a back slope has its occluder within 2 % of its
    range).  Judged by the vertex's own pixel alone the figures are 0.881 / 0.798 (exact line of sight 0.880 / 0.935)."""
    W, H, R = 3600, 600, 1200
    lat, lon = C1_EYES[1]
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    _, rng = h.render(-180., 180., lat=lat, lon=lon, znear=1., zfar=250000.)
    vis = h.viewshed([(lat, lon)])[0]
    z = h.mosaic().astype(np.float64)
    dems = h.context.dems
    cpd = dems.cells_per_deg
    vci = (lon - dems.origin_dem_lon_lat[0]) * cpd - dems.origin_dem_cellij[0]
    vcj = (lat - dems.origin_dem_lon_lat[1]) * cpd - dems.origin_dem_cellij[1]
    vz = h.move(lat, lon)
    cell = 6371000.0 * np.pi / 180.0 / cpd
    jj, ii = np.mgrid[0:2 * R, 0:2 * R].astype(np.float64)
    north = (jj - vcj) * cell
    east = (ii - vci) * cell * np.cos(np.radians(lat))
    d = np.hypot(east, north)
    sel = (d > 1000.) & (d < 5000.)
    hgt = z[sel] - vz
    az = np.degrees(np.arctan2(east[sel], north[sel]))
    el = np.degrees(np.arctan2(hgt, d[sel]))
    half_fov = 360.0 * H / W / 2
    x = np.floor((az + 180.) / 360. * W).astype(int) % W
    y_gl = np.floor((el / half_fov + 1.) / 2. * H).astype(int)
    keep = (y_gl >= 1) & (y_gl < H - 1)
    x, row = x[keep], H - 1 - y_gl[keep]
    seen = vis[sel][keep]
    el_row = np.radians(((H - 1 - row) + 0.5) / H * 2. * half_fov - half_fov)
    own = np.hypot(d[sel][keep], hgt[keep]) / np.cos(el_row)
    nb = np.stack([rng[row + a, (x + b) % W] for a in (-1, 0, 1) for b in (-1, 0, 1)])
    nearer = (nb > 0) & (nb < 0.98 * own)
    all_near, none_near = nearer.all(axis=0), ~nearer.any(axis=0)
    decides = all_near | none_near
    hidden_ok, visible_ok = all_near[~seen & decides].mean(), none_near[seen & decides].mean()
    print("renderer consistency: %d hidden, %d visible vertices, %.3f decidable; hidden with nearer terrain %.4f, "
          "visible without %.4f" % ((~seen).sum(), seen.sum(), decides.mean(), hidden_ok, visible_ok))
    assert (~seen & decides).sum() > 1000 and (seen & decides).sum() > 300
    assert hidden_ok >= 0.93 and visible_ok >= 0.92


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
        h = hz.horizonator(C1_LAT, C1_LON, 64, 16, dir_dems=tiles, render_radius_cells=300)
        views = [(C1_LAT + 0.011 * k, C1_LON - 0.009 * k) for k in range(-6, 7)]
        _, want = h.viewshed(views, counts=True)
        got = sharding.viewshed_counts_sharded(h, views)
        ok = np.array_equal(got.cpu().numpy(), want.astype(np.int32))
        got = sharding.viewshed_counts_sharded(h, views, root=0)
        if rank == 0:
            ok = ok and np.array_equal(got.cpu().numpy(), want.astype(np.int32))
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def test_nccl_sharded_counts_equal_one_gpu(tiles_c1):
    import torch
    import torch.multiprocessing as mp
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = min(n, 4)
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
