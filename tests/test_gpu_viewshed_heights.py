"""Viewshed heights on the GPU (horizonator_viewshed_heights*, include/horizonator-batch.h) against the oracle
(vs_oracle_r2_heights) bit for bit, at the mask's own edge cases (test_gpu_viewshed_edges.py: every mask width, eyes on
vertices and grid lines and in the outermost cells, explicit eye heights, flat-ground ties, missing tiles and voids,
refraction); against the kernel's own masks; the least over views on every path (per-view slices folded, direct
atomics, a second call, the host call); chunks; streams and interleaving with renders, masks and curvature changes;
argument handling; the minimum over two GPUs.  Run on the B200 box: pytest -m gpu."""
import ctypes as C
import os
import socket

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON
from oracle import vertex
from oracle.viewshed import unpack_mask
from oracle.viewshed_heights import r2_heights
from test_gpu_viewshed_edges import C2_LAT, C2_LON, PLACEMENTS, REFRACTIONS, Pair, _mixed_views, _place

pytestmark = pytest.mark.gpu

POISON = 0x5A5A5A5A
INF = 0x7F800000


def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test running without a CUDA device"
    return torch


def device_heights(p, views, least=None, per_view=True, stream=None):
    """One horizonator_viewshed_heights_device call; per-view heights into an array poisoned with POISON, returned as
    (n, N, N) uint32 patterns on the host (None with per_view=False); `least` a CUDA tensor folded into"""
    torch = _torch()
    d = torch.full((len(views), p.N, p.N), POISON, dtype=torch.int32, device="cuda") if per_view else None
    torch.cuda.synchronize()            # the context's own stream does not wait for torch's fills
    ok = p.hz.lib.horizonator_viewshed_heights_device(
        C.byref(p.h.context), len(views), p.h._eyes(views), d.data_ptr() if per_view else None,
        least.data_ptr() if least is not None else None, stream)
    assert ok, "horizonator_viewshed_heights_device refused the views"
    torch.cuda.synchronize()
    return d.cpu().numpy().view(np.uint32) if per_view else None


def inf_least(p):
    torch = _torch()
    return torch.full((p.N, p.N), INF, dtype=torch.int32, device="cuda")


def as_u32(t):
    return t.cpu().numpy().view(np.uint32)


def assert_same(got, want, v, what):
    """Bit patterns equal; on a difference: how many vertices, the first ones with both values, the eye"""
    if np.array_equal(got, want):
        return
    jj, ii = np.nonzero(got != want)
    g, w = got.view(np.float32), want.view(np.float32)
    first = ["(%d, %d) kernel %r oracle %r" % (i, j, float(g[j, i]), float(w[j, i])) for i, j in zip(ii[:6], jj[:6])]
    raise AssertionError("%s: %d vertices differ, eye cell (%r, %r), z %r; first %s"
                         % (what, len(ii), v["viewer_cell_i"], v["viewer_cell_j"], v["viewer_z"], "; ".join(first)))


def check(p, views, curvature=0., what="", stream=None):
    """Kernel against oracle for every view of one call, the heights' finiteness against the kernel's own masks at
    t = 1e30, and the call's least against the minimum of its views; returns the kernel's heights (uint32 patterns)"""
    least = inf_least(p)
    got = device_heights(p, views, least, stream=stream)
    inf_mask = unpack_mask(p.device(views, 1e30, stream=stream))
    for k, view in enumerate(views):
        p.o.move(view[0], view[1], view[4] if len(view) > 4 else None)
        v = p.o.viewer()
        want = r2_heights(p.vs, curvature=curvature).view(np.uint32)
        h = got[k].view(np.float32)
        print("%s view %d: eye cell (%r, %r), z %r, +0 %.5f, +inf %d, median of the rest %.2f m"
              % (what, k, v["viewer_cell_i"], v["viewer_cell_j"], v["viewer_z"], (got[k] == 0).mean(),
                 int((got[k] == INF).sum()), float(np.median(h[(h > 0) & np.isfinite(h)])) if ((h > 0) & np.isfinite(h)).any() else 0.))
        assert_same(got[k], want, v, "%s view %d" % (what, k))
        assert np.array_equal(np.isfinite(h), inf_mask[k]), "%s view %d: isfinite(heights) != mask at 1e30" % (what, k)
    assert np.array_equal(as_u32(least), got.min(axis=0)), "%s: least != the minimum of the views" % what
    return got


@pytest.fixture(scope="module")
def hz():
    import horizonator_b200
    return horizonator_b200


@pytest.fixture(scope="module")
def tiles_c2():
    from tools import synth
    return synth.config2_tiles(os.environ.get("HZ_BENCH_TILES", "/tmp/hz_tiles_c2"))


@pytest.fixture(scope="module")
def tiles_flat(tmp_path_factory):
    """No tiles at all: every height reads as 0"""
    return str(tmp_path_factory.mktemp("dems_none"))


@pytest.fixture(scope="module")
def pairs(hz):
    """pairs(tiles, R, srtm1=False): product/oracle pairs, one per (tiles, R, SRTM1) for the module (R None: 150 km)"""
    cache = {}

    def get(tiles, R, srtm1=False):
        key = (tiles, R, srtm1)
        if key not in cache:
            lat, lon = (C2_LAT, C2_LON) if srtm1 else (C1_LAT, C1_LON)
            cache[key] = Pair(hz, tiles, R, srtm1, lat, lon)
        return cache[key]
    yield get
    for p in cache.values():
        p.h.close()
        p.o.close()


C1_EYES = [(C1_LAT, C1_LON), (C1_LAT + 0.03, C1_LON - 0.02), (C1_LAT - 0.04, C1_LON + 0.05)]


# ---------------------------------------------------------------------------------------------- against the oracle

@pytest.mark.parametrize("refraction", [None, 0.13])
def test_c1_three_eyes(pairs, tiles_c1, refraction):
    p = pairs(tiles_c1, 1200)
    try:
        if refraction is not None:
            p.h.set_earth_curvature(True, refraction)
        c = vertex.curvature(True, refraction) if refraction is not None else 0.
        got = check(p, C1_EYES, curvature=c, what="C1 curvature %r" % refraction)
        assert 0.001 < (got == 0).mean() < 0.9
    finally:
        p.h.set_earth_curvature(False)


def test_c2_bench_viewpoint(pairs, tiles_c2):
    """C2 (SRTM1, N = 11716) at the bench viewpoint: one view's heights are 549 MB"""
    p = pairs(tiles_c2, None, True)
    assert p.N == 11716
    check(p, [(C2_LAT, C2_LON)], what="C2 bench viewpoint")


@pytest.mark.parametrize("where", ["centre", "corner"])
@pytest.mark.parametrize("R", [1, 2, 3, 15, 16, 17, 31, 33, 47, 300])
def test_every_mask_width(pairs, tiles_c1, R, where):
    p = pairs(tiles_c1, R)
    N = p.N
    view = (C1_LAT, C1_LON) if where == "centre" else p.view(("below", N - 1), 0.3)
    check(p, [view], what="N %d %s" % (N, where))


@pytest.mark.parametrize("name", PLACEMENTS)
@pytest.mark.parametrize("R", [300, 1200])
def test_eye_placements(pairs, tiles_c1, R, name):
    p = pairs(tiles_c1, R)
    view = _place(p, name)
    views = [view]
    if name in ("vertex", "vertical line", "horizontal line"):
        # an eye just under the ground, as for the masks
        v = p.o.viewer()
        i0, j0 = int(np.floor(v["viewer_cell_i"])), int(np.floor(v["viewer_cell_j"]))
        views.append(view[:2] + (0., 0., float(p.vs.heights[j0:j0 + 2, i0:i0 + 2].min()) - 0.25))
    check(p, views, what="R %d %s" % (R, name))


@pytest.mark.parametrize("R", [300, 1200])
def test_explicit_eye_heights(pairs, tiles_c1, R):
    p = pairs(tiles_c1, R)
    low = float(np.percentile(p.vs.heights, 10))
    views = [p.view(R - 0.3, R + 0.2, z) for z in (0., low, 9000.)] + [p.on_vertex(R + 20, R - 30, 0.)]
    got = check(p, views, what="R %d explicit z" % R)
    assert (got[2] == 0).mean() > 0.5


@pytest.mark.parametrize("R", [2, 17, 300])
def test_flat_ground_ties_everywhere(pairs, tiles_flat, R):
    """No tiles: every vertex is seen at the ground, from an eye on it (every slope 0, every comparison a tie) or 1 m
    up"""
    p = pairs(tiles_flat, R)
    N = p.N
    views = [p.view(R - 0.3, R + 0.2, 0.), p.view(0.5, ("below", N - 1), 0.), p.view(0.0, 0.0, 0.),
             p.view(R - 0.3, R + 0.2)]
    if R > 2:
        views.append(p.on_vertex(R + 5, R - 7, 0.))
    got = check(p, views, what="flat R %d" % R)
    assert (got == 0).all()


@pytest.mark.parametrize("R", [300, 1200])
def test_missing_and_empty_tiles(pairs, tiles_holes, R):
    p = pairs(tiles_holes, R)
    views = [(C1_LAT, C1_LON), p.view(R + 0.3, R - 0.6), p.view(0.5, 0.5), p.view(("below", p.N - 1), ("below", p.N - 1))]
    check(p, views, what="holes R %d" % R)


def test_voids_of_the_synthetic_tiles(pairs, tiles_c1):
    p = pairs(tiles_c1, 1200)
    jj, ii = np.nonzero(p.vs.heights == 0)
    k = np.argsort(np.hypot(ii - 1200, jj - 1200))[0]
    i, j = int(ii[k]), int(jj[k])
    views = [p.view(min(max(i + di, 0.5), 2398.5), min(max(j + dj, 0.5), 2398.5)) for di, dj in ((1.5, 0.5), (-3.5, -2.5))]
    check(p, views, what="void at (%d, %d)" % (i, j))


@pytest.mark.parametrize("refraction", REFRACTIONS)
def test_curvature(pairs, tiles_c1, refraction):
    p = pairs(tiles_c1, 1200)
    views = [(C1_LAT, C1_LON), p.on_vertex(1220, 1170), p.view(0.5, 2398.5)]
    try:
        p.h.set_earth_curvature(True, refraction)
        check(p, views, curvature=vertex.curvature(True, refraction), what="refraction %g" % refraction)
    finally:
        p.h.set_earth_curvature(False)


# ---------------------------------------------------------------------------------------------- least, chunks, host call

def test_least_on_every_path(hz, pairs, tiles_c1):
    """The least-only walk (atomics straight into least) equals the per-view slices folded by k_viewshed_least; a
    second call folds into the first; the host call folds into the caller's array and equals the device call"""
    torch = _torch()
    p = pairs(tiles_c1, 300)
    views = _mixed_views(p)
    a, b = views[:70], views[70:]
    la = inf_least(p)
    ha = device_heights(p, a, la)
    want_a = ha.min(axis=0)
    assert np.array_equal(as_u32(la), want_a)
    direct = inf_least(p)
    device_heights(p, a, direct, per_view=False)
    assert np.array_equal(as_u32(direct), want_a), "least-only path != per-view path"
    device_heights(p, b, direct, per_view=False)
    hb = device_heights(p, b)
    want = np.minimum(want_a, hb.min(axis=0))
    assert np.array_equal(as_u32(direct), want), "the second call did not fold into the first"
    assert (want == 0).any() and (want != 0).any()

    # host memory: min-folded into a caller's pattern (values >= +0, +inf and +0 among them), twice
    rs = np.random.default_rng(5)
    pattern = rs.exponential(20., (p.N, p.N)).astype(np.float32)
    pattern[rs.random((p.N, p.N)) < 0.3] = np.inf
    pattern[rs.random((p.N, p.N)) < 0.05] = 0.
    hl = pattern.copy()
    for rep in (1, 2):
        assert hz.lib.horizonator_viewshed_heights(C.byref(p.h.context), len(a), p.h._eyes(a), None, hl.ctypes.data)
        assert np.array_equal(hl.view(np.uint32), np.minimum(pattern.view(np.uint32), want_a)), rep
    hl = pattern.copy()
    assert hz.lib.horizonator_viewshed_heights(C.byref(p.h.context), len(b), p.h._eyes(b), None, hl.ctypes.data)
    assert np.array_equal(hl.view(np.uint32), np.minimum(pattern.view(np.uint32), hb.min(axis=0)))
    # per-view heights and least into host memory, and the Python wrappers
    hh = np.full((len(a), p.N, p.N), POISON, np.uint32)
    hl = pattern.copy()
    assert hz.lib.horizonator_viewshed_heights(C.byref(p.h.context), len(a), p.h._eyes(a), hh.ctypes.data, hl.ctypes.data)
    assert np.array_equal(hh, ha) and np.array_equal(hl.view(np.uint32), np.minimum(pattern.view(np.uint32), want_a))
    h2, l2 = p.h.viewshed_heights(a, least=True)
    assert np.array_equal(h2.view(np.uint32), ha) and np.array_equal(l2.view(np.uint32), want_a)
    assert np.array_equal(p.h.viewshed_least_height(a).view(np.uint32), want_a)
    t = torch.full((p.N, p.N), float("inf"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    p.h.viewshed_heights_device(a, d_least=t.data_ptr())
    assert np.array_equal(as_u32(t), want_a)


def test_the_first_least_call_of_a_context_folds_into_the_callers_least(hz, tiles_c1):
    """On a fresh context the host call's device least is allocated by this call"""
    p = Pair(hz, tiles_c1, 300, False, C1_LAT, C1_LON)
    try:
        views = _mixed_views(p)[:10]
        pattern = np.random.default_rng(9).exponential(20., (p.N, p.N)).astype(np.float32)
        hl = pattern.copy()
        assert hz.lib.horizonator_viewshed_heights(C.byref(p.h.context), len(views), p.h._eyes(views), None,
                                                   hl.ctypes.data)
        want = pattern.view(np.uint32)
        for v in views:
            p.o.move(v[0], v[1], v[4])
            want = np.minimum(want, r2_heights(p.vs).view(np.uint32))
        assert np.array_equal(hl.view(np.uint32), want)
    finally:
        p.h.close()
        p.o.close()


def test_100_views_equal_the_same_views_alone(pairs, tiles_c1):
    """chunks of 64 + 36"""
    p = pairs(tiles_c1, 300)
    views = _mixed_views(p)[:100]
    least = inf_least(p)
    batch = device_heights(p, views, least)
    for k, v in enumerate(views):
        assert np.array_equal(device_heights(p, [v])[0], batch[k]), k
    assert np.array_equal(as_u32(least), batch.min(axis=0))


def test_c2_host_call_in_scratch_chunks(hz, pairs, tiles_c2):
    """At C2 the host call's per-view scratch holds 3 views (2 GiB): 4 views go in chunks of 3 + 1"""
    p = pairs(tiles_c2, None, True)
    t = vertex.TILE_CELLS // 2 + 0.5
    views = [(C2_LAT, C2_LON), p.view(t, t), p.view(("below", p.N - 1), p.N // 2 + 0.3), (C2_LAT + 0.3, C2_LON - 0.4)]
    least = inf_least(p)
    dev = device_heights(p, views, least)
    hh = np.full((len(views), p.N, p.N), POISON, np.uint32)
    hl = np.full((p.N, p.N), np.inf, np.float32)
    assert hz.lib.horizonator_viewshed_heights(C.byref(p.h.context), len(views), p.h._eyes(views), hh.ctypes.data,
                                               hl.ctypes.data)
    for k in range(len(views)):
        assert np.array_equal(hh[k], dev[k]), k
    assert np.array_equal(hl.view(np.uint32), as_u32(least))


# ---------------------------------------------------------------------------------------------- streams, interleaving

def test_on_a_side_stream(pairs, tiles_c1):
    torch = _torch()
    p = pairs(tiles_c1, 300)
    views = _mixed_views(p)[:70]
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        check(p, views, what="side stream", stream=s.cuda_stream)


def test_interleaved_with_renders_masks_and_curvature(pairs, tiles_c1):
    """Heights between renders, mask calls and curvature toggles are the oracle's for the mode then current, and the
    renders and masks around them are what they are without heights calls in between"""
    torch = _torch()
    p = pairs(tiles_c1, 1200)
    views = [(C1_LAT, C1_LON), p.on_vertex(1220, 1170), p.view(("below", p.N - 1), 0.3)]
    W, H = 64, 16
    rviews = [(C1_LAT + 0.01 * k, C1_LON - 0.02 * k, -180., 180.) for k in range(3)]
    img = torch.zeros((len(rviews), H, W, 3), dtype=torch.uint8, device="cuda")
    rng = torch.zeros((len(rviews), H, W), dtype=torch.float32, device="cuda")
    c = vertex.curvature(True, 0.13)

    def render():
        torch.cuda.synchronize()
        p.h.render_batch_device(rviews, img.data_ptr(), rng.data_ptr())
        torch.cuda.synchronize()
        return img.cpu().numpy().copy(), rng.cpu().numpy().copy()

    try:
        img0, rng0 = render()
        masks0 = p.device(views, 1.7)
        check(p, views, what="after a render and a mask call")
        img1, rng1 = render()
        assert np.array_equal(img1, img0) and np.array_equal(rng1, rng0)
        assert np.array_equal(p.device(views, 1.7), masks0)
        p.h.set_earth_curvature(True, 0.13)
        check(p, views, curvature=c, what="curvature on")
        render()
        check(p, views, curvature=c, what="curvature on, after a render")
        p.h.set_earth_curvature(False)
        check(p, views, what="curvature off again")
        img2, rng2 = render()
        assert np.array_equal(img2, img0) and np.array_equal(rng2, rng0)
        assert np.array_equal(p.device(views, 1.7), masks0)
    finally:
        p.h.set_earth_curvature(False)


# ---------------------------------------------------------------------------------------------- arguments

def test_bad_arguments_write_nothing(hz, pairs, tiles_c1):
    torch = _torch()
    p = pairs(tiles_c1, 200)
    N, lib, ctx = p.N, hz.lib, C.byref(p.h.context)
    heights = torch.full((2, N, N), POISON, dtype=torch.int32, device="cuda")
    least = torch.full((N, N), POISON, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ok = [(C1_LAT, C1_LON)]
    outside = [(C1_LAT, C1_LON), (C1_LAT + 0.2, C1_LON)]                 # R = 200 cells = 0.167 degrees
    hp, lp = heights.data_ptr(), least.data_ptr()
    assert lib.horizonator_viewshed_heights_device(ctx, 0, p.h._eyes(ok), hp, lp, None)
    assert lib.horizonator_viewshed_heights_device(ctx, 0, None, hp, lp, None)
    assert not lib.horizonator_viewshed_heights_device(ctx, -1, p.h._eyes(ok), hp, lp, None)
    assert not lib.horizonator_viewshed_heights_device(ctx, 1, None, hp, lp, None)
    assert not lib.horizonator_viewshed_heights_device(ctx, 1, p.h._eyes(ok), None, None, None)
    assert not lib.horizonator_viewshed_heights_device(ctx, 2, p.h._eyes(outside), hp, lp, None)
    assert not lib.horizonator_viewshed_heights_device(ctx, 2, p.h._eyes(outside), None, lp, None)
    torch.cuda.synchronize()
    assert (heights == POISON).all().item() and (least == POISON).all().item()
    hh = np.full((2, N, N), POISON, np.uint32)
    hl = np.full((N, N), POISON, np.uint32)
    assert lib.horizonator_viewshed_heights(ctx, 0, p.h._eyes(ok), hh.ctypes.data, hl.ctypes.data)
    assert not lib.horizonator_viewshed_heights(ctx, -1, p.h._eyes(ok), hh.ctypes.data, hl.ctypes.data)
    assert not lib.horizonator_viewshed_heights(ctx, 1, None, hh.ctypes.data, hl.ctypes.data)
    assert not lib.horizonator_viewshed_heights(ctx, 1, p.h._eyes(ok), None, None)
    assert not lib.horizonator_viewshed_heights(ctx, 2, p.h._eyes(outside), hh.ctypes.data, hl.ctypes.data)
    assert not lib.horizonator_viewshed_heights(ctx, 2, p.h._eyes(outside), None, hl.ctypes.data)
    assert (hh == POISON).all() and (hl == POISON).all()
    with pytest.raises(RuntimeError):
        p.h.viewshed_least_height(outside)


# ---------------------------------------------------------------------------------------------- two GPUs

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
        want = h.viewshed_least_height(views).view(np.uint32)
        got = sharding.viewshed_least_height_sharded(h, views)
        ok = np.array_equal(got.cpu().numpy().view(np.uint32), want)
        got = sharding.viewshed_least_height_sharded(h, views, root=0)
        if rank == 0:
            ok = ok and np.array_equal(got.cpu().numpy().view(np.uint32), want)
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def test_nccl_sharded_least_equals_one_gpu(tiles_c1):
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
