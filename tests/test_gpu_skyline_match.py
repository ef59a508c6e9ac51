"""Skylines and their match against an observed skyline on the GPU (horizonator_skyline_match*,
include/horizonator-batch.h): rows and range against horizon_profile_device() of the same renders' range images, scores
against the host restatement of the rule (oracle/skyline_match.py) on the GPU's own rows, the host call against the
device call, rendering untouched, an end-to-end search for a photo's eye and heading, argument handling, C2 at the
bench viewpoint, sharded over NCCL.  Run on the B200 box: pytest -m gpu."""
import ctypes as C
import os
import socket

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON
from oracle import skyline_match as om

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hz():
    import horizonator_b200
    return horizonator_b200


def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test running without a CUDA device"
    return torch


# ---------------------------------------------------------------------------------------------- inputs

def _views_c1(n, seed=11):
    """n views: full circle, 90 degrees, 5-degree zooms, 120 and 60 degrees, explicit eye heights, eyes near the
    square's edge."""
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


def _profile(h, views):
    """(rows, range) of horizon_profile_device() on render_batch_device() range images of the views"""
    torch = _torch()
    n, W, H = len(views), h.width, h.height
    rng = torch.empty((n, H, W), dtype=torch.float32, device="cuda")
    h.render_batch_device(views, 0, rng.data_ptr())
    rows = torch.empty((n, W), dtype=torch.int32, device="cuda")
    rr = torch.empty((n, W), dtype=torch.float32, device="cuda")
    h.horizon_profile_device(rng.data_ptr(), n, rows.data_ptr(), rr.data_ptr())
    torch.cuda.synchronize()
    return rows.cpu().numpy(), rr.cpu().numpy()


def _device(h, views, smp=None, clip=8., wrap=True, rows=True, rng=True, scores=True, stream=0):
    """(rows, range, scores) of one skyline_match_device call, None where not asked for; the outputs start poisoned"""
    torch = _torch()
    n, W = len(views), h.width
    r = torch.full((n, W), 77, dtype=torch.int32, device="cuda") if rows else None
    g = torch.full((n, W), 7.0, dtype=torch.float32, device="cuda") if rng else None
    s = torch.full((n, W), 7.0, dtype=torch.float32, device="cuda") if scores else None
    d_smp = torch.as_tensor(smp.view(np.int32).reshape(-1, 2), device="cuda") if scores else 0
    h.skyline_match_device(views, d_smp, s if scores else 0, r if rows else 0, g if rng else 0, clip_rows=clip,
                           wrap=wrap, stream=stream, m=len(smp) if scores else 0)
    torch.cuda.synchronize()
    return tuple(t.cpu().numpy() if t is not None else None for t in (r, g, s))


def _random_samples(W, H, m, seed):
    rs = np.random.default_rng(seed)
    dx = rs.integers(-3 * W // 2, 3 * W // 2, m)
    y = rs.uniform(-20, H + 20, m)
    y[::5] = rs.integers(0, H, len(y[::5])) - 0.5            # exactly on rendered edges
    return om.samples(np.stack([dx, y], axis=1))


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ---------------------------------------------------------------------------------------------- 1
@pytest.mark.parametrize("mode", [None, "profiled", "seam_wrap", "lod", "curvature"])
def test_rows_and_range_equal_the_horizon_profile(hz, tiles_c1, mode):
    h = _c1(hz, tiles_c1, 600, 150, mode)
    base = _views_c1(24)
    # the 24 views, then the same turned by 0.37 degrees per round
    views = [(v[0], v[1], float(np.float32(v[2] + 0.37 * (k // 24))), float(np.float32(v[3] + 0.37 * (k // 24))), v[4])
             for k, v in ((k, base[k % 24]) for k in range(300))]
    for n in (1, 7, 64, 65, 300):
        want_rows, want_rng = _profile(h, views[:n])
        rows, rng, _ = _device(h, views[:n], scores=False)
        assert np.array_equal(rows, want_rows), (mode, n)
        assert np.array_equal(_bits(rng), _bits(want_rng)), (mode, n)
    assert (rows >= 0).mean() > 0.25, mode                   # terrain in a good share of the columns
    hr, hg = h.skyline(views)
    assert np.array_equal(hr, rows) and np.array_equal(_bits(hg), _bits(rng))
    if mode == "profiled":
        assert h.profile_read()["renders"] > 0
        h.profile(False)


# ---------------------------------------------------------------------------------------------- 2
def test_scores_equal_the_host_rule_on_the_gpus_rows(hz, tiles_c1):
    W, H = 1200, 300
    h = _c1(hz, tiles_c1, W, H)
    views = _views_c1(24)
    for m in (1, 37, 600, 3600):
        smp = _random_samples(W, H, m, seed=m)
        for wrap in (True, False):
            for clip in (8.0, 2.5):
                rows, _, scores = _device(h, views, smp, clip=clip, wrap=wrap, rng=False)
                want = om.scores(rows, smp, clip, wrap)
                assert np.array_equal(_bits(scores), _bits(want)), (m, wrap, clip)
                assert 0.0 <= scores.min() and scores.max() <= clip


# ---------------------------------------------------------------------------------------------- 3
def test_host_call_device_call_and_output_subsets_agree(hz, tiles_c1):
    W, H = 900, 200
    h = _c1(hz, tiles_c1, W, H)
    views = _views_c1(70, seed=3)
    smp = _random_samples(W, H, 300, seed=5)
    rows, rng, scores = _device(h, views, smp, clip=6.0, wrap=True)
    r_only, _, _ = _device(h, views, rng=False, scores=False)
    _, _, s_only = _device(h, views, smp, clip=6.0, wrap=True, rows=False, rng=False)
    assert np.array_equal(r_only, rows) and np.array_equal(_bits(s_only), _bits(scores))
    hs, hr = h.skyline_match(views, smp, clip_rows=6.0, wrap=True, rows=True)
    assert np.array_equal(hr, rows) and np.array_equal(_bits(hs), _bits(scores))
    assert np.array_equal(_bits(h.skyline_match(views, smp, clip_rows=6.0)), _bits(scores))
    hr2, hg2 = h.skyline(views)
    assert np.array_equal(hr2, rows) and np.array_equal(_bits(hg2), _bits(rng))
    # (dx, y) pairs work as well as the structured array
    pairs = [(int(a), float(b)) for a, b in zip(smp["dx"], smp["y"])]
    assert np.array_equal(_bits(h.skyline_match(views[:5], pairs, clip_rows=6.0)), _bits(scores[:5]))


# ---------------------------------------------------------------------------------------------- 4
def test_rendering_is_untouched(hz, tiles_c1):
    torch = _torch()
    W, H = 1000, 200
    h = _c1(hz, tiles_c1, W, H)
    views = _views_c1(20, seed=8)
    smp = _random_samples(W, H, 200, seed=9)
    st = torch.cuda.Stream()
    s = st.cuda_stream
    img = [torch.empty((20, H, W, 3), dtype=torch.uint8, device="cuda") for _ in range(3)]
    rng = [torch.empty((20, H, W), dtype=torch.float32, device="cuda") for _ in range(3)]
    rows = [torch.empty((20, W), dtype=torch.int32, device="cuda") for _ in range(2)]
    sc = torch.empty((20, W), dtype=torch.float32, device="cuda")
    d_smp = torch.as_tensor(smp.view(np.int32).reshape(-1, 2), device="cuda")
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        h.render_batch_device(views, img[0].data_ptr(), rng[0].data_ptr(), s)
        h.skyline_match_device(views, d_smp, sc, rows[0], stream=s)
        h.render_batch_device(views, img[1].data_ptr(), rng[1].data_ptr(), s)
        h.skyline_match_device(views[::-1], d_smp, 0, rows[1], stream=s)
        h.render_batch_device(views, 0, rng[2].data_ptr(), s)
        h.render_batch_device(views, img[2].data_ptr(), 0, s)
    torch.cuda.synchronize()
    for k in (1, 2):
        assert torch.equal(img[k], img[0]) and torch.equal(rng[k].view(torch.int32), rng[0].view(torch.int32)), k
    want_rows, _ = _profile(h, views)
    assert np.array_equal(rows[0].cpu().numpy(), want_rows)
    assert np.array_equal(rows[1].cpu().numpy(), want_rows[::-1])


# ---------------------------------------------------------------------------------------------- 5
def _grid(lat0, lon0, step, k_lat, k_lon):
    """8 x 8 candidate eyes, the true one (lat0, lon0) at grid position (k_lat, k_lon)"""
    return [(float(np.float32(lat0 + (i - k_lat) * step)), float(np.float32(lon0 + (j - k_lon) * step)))
            for i in range(8) for j in range(8)]


def test_search_finds_the_eye_and_heading(hz, tiles_c1):
    W, H = 3600, 600
    h = _c1(hz, tiles_c1, W, H)
    p = 360.0 / W
    eyes = _grid(C1_LAT + 0.05, C1_LON - 0.07, 0.02, 3, 5)
    true = 3 * 8 + 5
    cand = [(la, lo, -180.0, 180.0) for la, lo in eyes]
    # exact case: 600 columns of the true eye's own skyline, from column c0 on
    rows, _ = h.skyline([cand[true]])
    c0 = 1500
    cols = [(c0 + d) % W for d in range(600)]
    smp = om.samples([(d, rows[0, c] - 0.5) for d, c in enumerate(cols) if rows[0, c] >= 0])
    assert len(smp) > 400
    best = h.locate(cand, smp, top=5)
    assert best[0][0] == true and best[0][2] == 0.0
    assert abs(best[0][1] - (-180.0 + (c0 + 0.5) * p)) < 1e-9
    assert best[1][2] > 0.0
    # realistic case: the "photo" is a 60-degree view of another size (its window 0.3 column off the search's column
    # grid), its skyline turned into angles relative to its centre and then into samples
    Wp, Hp, fov = 600, 400, 60.0
    hp = _c1(hz, tiles_c1, Wp, Hp)
    az0 = float(np.float32(-180.0 + 1400.3 * p))
    photo_view = (cand[true][0], cand[true][1], az0, float(np.float32(az0 + fov)))
    heading = (photo_view[2] + photo_view[3]) / 2.
    prow, _ = hp.skyline([photo_view])
    pp = (photo_view[3] - photo_view[2]) / Wp
    c = np.nonzero(prow[0] >= 0)[0]
    assert len(c) > Wp // 2
    rel = (photo_view[2] + (c + 0.5) * pp) - heading
    el = ((Hp - 1) / 2. - (prow[0, c] - 0.5)) * pp
    smp2 = h.skyline_samples(rel, el, 360.0)
    scores = h.skyline_match(cand, smp2)
    best = h.locate(cand, smp2, top=3)
    print("photo search:", best, "truth", (true, heading), "true eye's best", (int(scores[true].argmin()), float(scores[true].min())))
    assert best[0][0] == true
    assert abs(best[0][1] - heading) <= p + 1e-6


# ---------------------------------------------------------------------------------------------- 6
def test_invalid_arguments_write_nothing(hz, tiles_c1):
    torch = _torch()
    h = _c1(hz, tiles_c1, 64, 16)
    ctx, lib = C.byref(h.context), hz.lib
    views = h._views([(C1_LAT, C1_LON, 0., 90.)] * 2)
    smp = torch.zeros((4, 2), dtype=torch.int32, device="cuda")
    rows = torch.full((2, 64), 77, dtype=torch.int32, device="cuda")
    rng = torch.full((2, 64), 7.0, dtype=torch.float32, device="cuda")
    sc = torch.full((2, 64), 7.0, dtype=torch.float32, device="cuda")
    S, R, G, Q = smp.data_ptr(), rows.data_ptr(), rng.data_ptr(), sc.data_ptr()
    f = lib.horizonator_skyline_match_device
    assert not f(ctx, -1, views, R, G, 4, S, 8.0, True, Q, None)
    assert not f(ctx, 2, None, R, G, 4, S, 8.0, True, Q, None)
    assert not f(ctx, 2, views, None, None, 4, S, 8.0, True, None, None)     # nothing asked for
    assert not f(ctx, 2, views, R, G, 0, S, 8.0, True, Q, None)              # scores without samples
    assert not f(ctx, 2, views, R, G, -3, S, 8.0, True, Q, None)
    assert not f(ctx, 2, views, R, G, 4, None, 8.0, True, Q, None)
    for clip in (0.0, -1.0, float("inf"), float("nan")):
        assert not f(ctx, 2, views, R, G, 4, S, clip, True, Q, None), clip
    assert not f(ctx, 2, views, R, G, 4, S + 4, 8.0, True, Q, None)          # misaligned samples
    assert not f(ctx, 2, views, R + 2, G, 4, S, 8.0, True, Q, None)          # misaligned rows
    assert f(ctx, 0, views, R, G, 4, S, 8.0, True, Q, None)
    assert f(ctx, 0, None, None, None, 0, None, 0.0, True, None, None)
    torch.cuda.synchronize()
    assert (rows == 77).all().item() and (rng == 7.0).all().item() and (sc == 7.0).all().item()
    hr = np.full((2, 64), 77, np.int32)
    hs = np.full((2, 64), 7.0, np.float32)
    hsmp = np.zeros(4, om.SAMPLE_DTYPE)
    g = lib.horizonator_skyline_match
    assert not g(ctx, -1, views, hr.ctypes.data, None, 4, hsmp.ctypes.data, 8.0, True, hs.ctypes.data)
    assert not g(ctx, 2, views, None, None, 4, hsmp.ctypes.data, 8.0, True, None)
    assert not g(ctx, 2, views, hr.ctypes.data, None, 0, hsmp.ctypes.data, 8.0, True, hs.ctypes.data)
    assert not g(ctx, 2, views, hr.ctypes.data, None, 4, None, 8.0, True, hs.ctypes.data)
    assert not g(ctx, 2, views, hr.ctypes.data, None, 4, hsmp.ctypes.data, 0.0, True, hs.ctypes.data)
    assert g(ctx, 0, views, hr.ctypes.data, None, 4, hsmp.ctypes.data, 8.0, True, hs.ctypes.data)
    assert (hr == 77).all() and (hs == 7.0).all()
    # rows only ignores the samples' arguments; a valid call does write
    assert g(ctx, 2, views, hr.ctypes.data, None, 0, None, 0.0, True, None) and not (hr == 77).all()
    assert g(ctx, 2, views, None, None, 4, hsmp.ctypes.data, 8.0, True, hs.ctypes.data) and not (hs == 7.0).all()


# ---------------------------------------------------------------------------------------------- 7
def test_c2_at_the_bench_viewpoint(hz):
    import bench
    from tools import synth
    C2 = bench.C2
    tiles = synth.config2_tiles(os.environ.get("HZ_BENCH_TILES", "/tmp/hz_tiles_c2"))
    h = hz.horizonator(C2["lat"], C2["lon"], C2["W"], C2["H"], SRTM1=True, dir_dems=tiles, render_radius_m=C2["radius_m"])
    h.set_zextents(C2["znear"], C2["zfar"])
    views = [(C2["lat"], C2["lon"], C2["az0"] + 0.7 * k, C2["az1"] + 0.7 * k) for k in range(256)]
    want_rows, want_rng = _profile(h, views)
    smp = _random_samples(C2["W"], C2["H"], 600, seed=12)
    rows, rng, scores = _device(h, views, smp, clip=8.0, wrap=True)
    assert np.array_equal(rows, want_rows) and np.array_equal(_bits(rng), _bits(want_rng))
    pick = list(range(0, 256, 16))
    assert np.array_equal(_bits(scores[pick]), _bits(om.scores(rows[pick], smp, 8.0, True)))


# ---------------------------------------------------------------------------------------------- 8
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
        smp = _random_samples(800, 200, 150, seed=4)
        want = h.skyline_match(views, smp, clip_rows=5.0)
        got = sharding.skyline_match_sharded(h, views, smp, clip_rows=5.0)
        q.put((rank, bool(np.array_equal(_bits(got.cpu().numpy()), _bits(want)))))
    finally:
        dist.destroy_process_group()


def test_nccl_sharded_scores_equal_one_gpu(tiles_c1):
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
