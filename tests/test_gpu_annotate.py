"""Labels of points of interest on the GPU (horizonator_annotate_batch*, include/horizonator-batch.h) against the host
restatement of the rule (oracle/annotate.py) on the range images of the same call; labels-only against labels with
outputs, batches against lone views, the host call against the device call; rendering untouched; the command-line
tool's --labels; the opt-in modes; C2 at the bench viewpoint; argument handling; sharded over NCCL.
Run on the B200 box: pytest -m gpu."""
import ctypes as C
import json
import math
import os
import socket
import subprocess

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON
from oracle import annotate as oa

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "horizonator_b200", "bin", "horizonator-standalone")


@pytest.fixture(scope="module")
def hz():
    import horizonator_b200
    return horizonator_b200


def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test running without a CUDA device"
    return torch


# ---------------------------------------------------------------------------------------------- inputs

def _views_c1():
    """24 views: (nearly) full circle, 90 degrees, 5-degree zooms, explicit eye heights, eyes near the square's edge.
    (A window of exactly 360 degrees makes horizonator_project() fail for every POI: horizonator-batch.h.)"""
    rs = np.random.default_rng(11)
    v = []
    for k in range(24):
        lat, lon = C1_LAT + rs.uniform(-0.25, 0.25), C1_LON + rs.uniform(-0.25, 0.25)
        kind = k % 6
        if kind == 0:
            az0 = rs.uniform(-180, 180); az1 = az0 + 359.9
        elif kind == 1:
            az0 = rs.uniform(-180, 180); az1 = az0 + 90.0
        elif kind == 2:
            az0 = rs.uniform(-180, 180); az1 = az0 + 5.0
        elif kind == 3:
            az0 = rs.uniform(-180, 180); az1 = az0 + 120.0
        elif kind == 4:
            lat, lon = C1_LAT + 0.93, C1_LON - 0.94 + 0.05 * k / 24      # near the north-west edge of the R=1200 square
            az0 = rs.uniform(-180, 180); az1 = az0 + 180.0
        else:
            az0 = rs.uniform(-180, 180); az1 = az0 + 60.0
        z = float(rs.uniform(1500, 3000)) if k % 4 == 3 else -1.0     # explicit eye heights
        v.append((float(np.float32(lat)), float(np.float32(lon)), float(np.float32(az0)), float(np.float32(az1)), z))
    return v


def _eye(h, view):
    """the eye height the library uses for a view: viewer_z as the float it travels as, or horizonator_move()'s"""
    return float(np.float32(view[4])) if len(view) > 4 and view[4] >= 0 else h.move(view[0], view[1])


def _skyline(h, views, ranges, per_view, seed):
    """Points on the rendered skyline (the topmost terrain pixel of a column, 2..30 km away), as lat, lon, ele."""
    W, H = h.width, h.height
    rs = np.random.default_rng(seed)
    out = []
    la, lo = C.c_float(), C.c_float()
    for view, rng in zip(views, ranges):
        lat, lon, az0, az1 = view[:4]
        eye = _eye(h, view)
        top = np.argmax(rng > 0, axis=0)
        cols = [c for c in range(3, W - 3) if top[c] > 8 and 2000. < rng[top[c], c] < 30000.]
        for c in rs.choice(cols, min(per_view, len(cols)), replace=False):
            y = int(top[c])
            el = math.radians((1 - (2 * y + 1) / H) * (az1 - az0) / (2 * (W / H)))
            # reported range = slant / cos(el) (reference quirk Q1): horizontal distance = range * cos(el)^2
            dist = float(rng[y, c]) * math.cos(el) ** 2
            assert _unproject(h, la, lo, int(c), y, dist, lat, lon, az0, az1)
            out.append((la.value, lo.value, eye + dist * math.tan(el)))
    return np.array(out, np.float64).reshape(-1, 3)


def _unproject(h, la, lo, x, y, dist, lat, lon, az0, az1):
    """horizonator_unproject() of pixel (x, y) at horizontal distance `dist` of a view of h's size"""
    import horizonator_b200 as hz
    return hz.lib.horizonator_unproject(C.byref(la), C.byref(lo), x, y, -1., dist, float(np.float32(lat)),
                                        math.cos(math.radians(float(np.float32(lat)))), float(np.float32(lon)),
                                        az0, az1, h.width, h.height)


def _pois_c1(h, views, ranges):
    from tools.pois import summits
    rs = np.random.default_rng(5)
    s = summits(h, 900, seed=1)
    sky = _skyline(h, views[:6], ranges[:6], 80, seed=2)
    # near the terrain, a little above or below it
    z = h.mosaic()
    N = z.shape[0]
    from tools.pois import vertex_latlon
    i, j = rs.integers(0, N, 500), rs.integers(0, N, 500)
    lat, lon = vertex_latlon(h, i, j)
    near = np.stack([lat, lon, z[j, i] + rs.uniform(-40, 150, 500)], axis=1)
    special = []
    for k in range(20):
        special.append((C1_LAT + 0.1 + 0.01 * k, C1_LON, -5000.0))                 # buried
        special.append((C1_LAT + 0.001 * (k % 3), C1_LON + 0.0001 * k, 1500.0))    # too close
        special.append((C1_LAT + 1.5 + 0.01 * k, C1_LON, 3000.0))                 # too far
        special.append((C1_LAT - 0.2, C1_LON + 0.01 * k, 8000.0))                  # high up: outside the window
    return np.concatenate([s, sky, near, np.array(special)], axis=0)


def _annotate_device(h, views, pois, images=False, ranges=True):
    """-> (labels (n, m) LABEL_DTYPE, ranges (n, H, W) or None, images or None) of one annotate_batch_device call."""
    torch = _torch()
    n, W, H = len(views), h.width, h.height
    p = torch.as_tensor(np.ascontiguousarray(pois, np.float64), device="cuda")
    lab = torch.full((n, len(pois), 4), 7.0, dtype=torch.float32, device="cuda")
    rng = torch.empty((n, H, W), dtype=torch.float32, device="cuda") if ranges else None
    img = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda") if images else None
    h.annotate_device(views, p, lab, img.data_ptr() if images else 0, rng.data_ptr() if ranges else 0)
    torch.cuda.synchronize()
    out = lab.cpu().numpy().view(oa.LABEL_DTYPE)[..., 0]
    return out, (rng.cpu().numpy() if ranges else None), (img.cpu().numpy() if images else None)


def _ulp_close(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return np.abs(a.astype(np.float64) - b.astype(np.float64)) <= np.spacing(np.abs(b)).astype(np.float64)


def _ambiguous(o):
    """POIs whose host projection sits within 1e-9 of a rounding or comparison boundary of the rule (x at a half-integer:
    lround; y at a half-integer or an integer: lround and the y + d tests; range at a gate): there the device's atan2
    (libdevice), a last bit away from glibc's, may decide otherwise.  Exactly on a boundary is not ambiguous: a POI at
    the eye's height has y = H/2 - 0.5 exactly on both sides (atan2(0, d) = 0)."""
    def near(v, at):
        f = np.abs(v - np.floor(v) - at)
        return (f > 0) & (f < 1e-9)
    amb = near(o.x, 0.5) | near(o.y, 0.5) | near(o.y, 0.0) | near(o.y, 1.0)
    amb |= (np.abs(o.range - 500.0) < 1e-6) | (np.abs(o.range - 100000.0) < 1e-6)
    return amb & ~np.isnan(o.x)


def _compare_with_oracle(hz, h, views, pois, labels, ranges, what):
    """Test 1's comparison: every decision and offset equal, x / y / range_m within one float ulp, rendered ranges
    equal.  Returns the number of visible (view, POI) pairs."""
    project = hz.lib.horizonator_project
    visible = 0
    for k, v in enumerate(views):
        o = oa.annotate_view(project, ranges[k], pois, v[0], v[1], _eye(h, v), v[2], v[3])
        got, want = labels[k], o.labels
        amb = _ambiguous(o)
        if amb.any():
            print(what, "view", k, "POIs at a rounding boundary (not compared):", np.nonzero(amb)[0].tolist())
        ok = ~amb
        outside = np.isnan(o.x)
        assert (got.view(np.float32).reshape(-1, 4)[outside & ok] == -1.0).all(), (what, k)
        ins = ~outside & ok
        g_vis, w_vis = got["range_rendered_m"] > 0, o.visible
        bad = np.nonzero((g_vis != w_vis) & ins)[0]
        assert len(bad) == 0, (what, k, bad[:10], got[bad[:5]], want[bad[:5]])
        for f in ("x", "y", "range_m"):
            close = _ulp_close(got[f][ins], want[f][ins])
            assert close.all(), (what, k, f, np.nonzero(~close)[0][:10], got[f][ins][~close][:5], want[f][ins][~close][:5])
        # the search offset: y - projected y is exactly `best` (integer) on both sides
        vis = ins & w_vis
        assert np.array_equal(np.rint(got["y"][vis].astype(np.float64) - o.y[vis]), o.best[vis].astype(np.float64)), (what, k)
        assert np.array_equal(got["range_rendered_m"][ins], want["range_rendered_m"][ins]), (what, k)
        visible += int(vis.sum())
    return visible


# ---------------------------------------------------------------------------------------------- 1
def test_matches_the_host_rule_on_the_same_calls_range_images(hz, tiles_c1):
    W, H = 1200, 300
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=1200)
    h.set_zextents(100., 120000.)
    views = _views_c1()
    _, first = h.render_batch(views[:6], return_image=False)
    pois = _pois_c1(h, views, first)
    assert 1500 <= len(pois) <= 2500
    labels, ranges, _ = _annotate_device(h, views, pois)
    visible = _compare_with_oracle(hz, h, views, pois, labels, ranges, "c1")
    print("c1: %d views x %d POIs, %d visible" % (len(views), len(pois), visible))
    assert visible >= 300


# ---------------------------------------------------------------------------------------------- 2
@pytest.mark.parametrize("profiled", [False, True])
def test_labels_only_host_call_and_batches_agree(hz, tiles_c1, profiled):
    W, H = 600, 150
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=1200)
    h.set_zextents(100., 120000.)
    rs = np.random.default_rng(21)
    views = [(C1_LAT + rs.uniform(-0.3, 0.3), C1_LON + rs.uniform(-0.3, 0.3), a, a + rs.choice([359.9, 90., 20.]),
              -1. if k % 5 else 2500.) for k, a in enumerate(rs.uniform(-180, 180, 300))]
    from tools.pois import summits
    pois = summits(h, 500, seed=3)
    if profiled:
        h.profile(True)
    with_ranges, _, _ = _annotate_device(h, views[:65], pois, ranges=True)
    only, _, _ = _annotate_device(h, views[:65], pois, ranges=False)
    assert np.array_equal(only.view(np.uint32), with_ranges.view(np.uint32))
    host = h.annotate(views[:65], pois)
    assert host.shape == (65, len(pois)) and np.array_equal(host.view(np.uint32), only.view(np.uint32))
    assert (only["range_rendered_m"] > 0).sum() > 100
    lone = np.stack([_annotate_device(h, [v], pois, ranges=False)[0][0] for v in views])
    for n in (1, 7, 64, 65, 300):
        got, _, _ = _annotate_device(h, views[:n], pois, ranges=False)
        assert np.array_equal(got.view(np.uint32), lone[:n].view(np.uint32)), n
    assert np.array_equal(h.annotate(views, pois).view(np.uint32), lone.view(np.uint32))
    if profiled:
        assert h.profile_read()["renders"] > 0
        h.profile(False)


# ---------------------------------------------------------------------------------------------- 3
def test_rendering_is_untouched(hz, tiles_c1):
    torch = _torch()
    W, H = 1000, 200
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=1200)
    views = _views_c1()[:20]
    from tools.pois import summits
    pois = summits(h, 300, seed=4)
    _, rng_a, img_a = _annotate_device(h, views, pois, images=True, ranges=True)
    img = torch.empty((len(views), H, W, 3), dtype=torch.uint8, device="cuda")
    rng = torch.empty((len(views), H, W), dtype=torch.float32, device="cuda")
    h.render_batch_device(views, img.data_ptr(), rng.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(img.cpu().numpy(), img_a)
    assert np.array_equal(rng.cpu().numpy().view(np.uint32), rng_a.view(np.uint32))
    # images only, too
    _, _, img_b = _annotate_device(h, views, pois, images=True, ranges=False)
    assert np.array_equal(img_b, img_a)


# ---------------------------------------------------------------------------------------------- 4
def test_matches_the_command_line_tool(hz, tiles_c1, tmp_path):
    W, H, zfar = 1200, 300, 40000.
    lat, lon = 35.125, -116.875                                   # exact floats: both sides take the same inputs
    az_c, az_r = 30.0, 60.0
    # the tool's pixel-centre convention, in float as there
    az_r_f = np.float32(az_r) + np.float32(np.float32(2. * az_r / float(np.float32(W - 1))) / np.float32(2.))
    az0, az1 = float(np.float32(az_c) - az_r_f), float(np.float32(az_c) + az_r_f)
    h = hz.horizonator(lat, lon, W, H, dir_dems=tiles_c1, render_radius_m=zfar)
    h.set_zextents(100., zfar)
    view = (lat, lon, az0, az1)
    _, first = h.render_batch([view], return_image=False)
    from tools.pois import summits
    pois = np.concatenate([summits(h, 400, seed=6), _skyline(h, [view], first, 60, seed=7)])
    names = ["p%d" % i for i in range(len(pois))]
    csv = tmp_path / "pois.csv"
    csv.write_text("# name,lat,lon,ele\n" + "".join("%s,%r,%r,%r\n" % (nm, float(a), float(b), float(c))
                                                   for nm, (a, b, c) in zip(names, pois)))
    out = tmp_path / "labels.json"
    r = subprocess.run([CLI, "--width", str(W), "--height", str(H), "--zfar", str(zfar), "--dirdems", tiles_c1,
                        "--image", str(tmp_path / "o.png"), "--pois", str(csv), "--labels", str(out),
                        repr(lat), repr(lon), repr(az_c), repr(az_r)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    cli = {d["name"]: d for d in json.load(open(out))}
    lab = h.annotate([view], pois)[0]
    mine = {nm: lab[i] for i, nm in enumerate(names) if lab["range_rendered_m"][i] > 0}
    assert len(mine) >= 30
    assert set(mine) == set(cli)
    for nm, d in cli.items():
        g = mine[nm]
        for f, digits in (("x", 3), ("y", 3), ("range_m", 1), ("range_rendered_m", 1)):
            v = float(g[f])
            tol = 0.5 * 10.0 ** -digits + 2 * float(np.spacing(np.float32(abs(v))))
            assert abs(v - d[f]) <= tol, (nm, f, v, d[f])


# ---------------------------------------------------------------------------------------------- 5
@pytest.mark.parametrize("mode", ["seam_wrap", "lod"])
def test_opt_in_modes(hz, tiles_c1, mode):
    W, H = 1200, 300
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=1200)
    h.set_zextents(100., 120000.)
    if mode == "seam_wrap":
        h.set_seam_wrap(True)
    else:
        h.set_lod(1.0)
    views = _views_c1()[:12]
    _, first = h.render_batch(views[:6], return_image=False)
    pois = _pois_c1(h, views, first)
    labels, ranges, _ = _annotate_device(h, views, pois)
    visible = _compare_with_oracle(hz, h, views, pois, labels, ranges, mode)
    print(mode, "visible", visible)
    assert visible >= 150


# ---------------------------------------------------------------------------------------------- 6
def test_c2_at_the_bench_viewpoint(hz):
    import bench
    from tools import synth
    from tools.pois import summits
    C2 = bench.C2
    tiles = synth.config2_tiles(os.environ.get("HZ_BENCH_TILES", "/tmp/hz_tiles_c2"))
    h = hz.horizonator(C2["lat"], C2["lon"], C2["W"], C2["H"], SRTM1=True, dir_dems=tiles, render_radius_m=C2["radius_m"])
    h.set_zextents(C2["znear"], C2["zfar"])
    # the bench's window less a tenth of a degree (exactly 360 degrees projects nothing), turned by 0.7 degrees per view
    views = [(C2["lat"], C2["lon"], C2["az0"] + 0.7 * k, C2["az1"] - 0.1 + 0.7 * k) for k in range(256)]
    pois = summits(h, 10000, seed=9)
    labels, ranges, _ = _annotate_device(h, views, pois)
    assert labels.shape == (256, 10000)
    pick = list(range(0, 256, 16))
    visible = _compare_with_oracle(hz, h, [views[k] for k in pick], pois, labels[pick], ranges[pick], "c2")
    # summits of the rough synthetic C2 terrain are mostly hidden behind nearer ridges: 55 visible pairs were measured
    print("c2: visible in 16 views", visible)
    assert visible >= 30


# ---------------------------------------------------------------------------------------------- 7
def test_invalid_arguments_write_nothing(hz, tiles_c1):
    torch = _torch()
    h = hz.horizonator(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_c1, render_radius_cells=200)
    ctx, lib = C.byref(h.context), hz.lib
    views = h._views([(C1_LAT, C1_LON, 0., 90.)] * 2)
    p = torch.tensor([[C1_LAT + 0.05, C1_LON, 500.]] * 3, dtype=torch.float64, device="cuda")
    lab = torch.full((2, 3, 4), 7.0, dtype=torch.float32, device="cuda")
    rng = torch.full((2, 16, 64), 7.0, dtype=torch.float32, device="cuda")
    P, L, R = p.data_ptr(), lab.data_ptr(), rng.data_ptr()
    f = lib.horizonator_annotate_batch_device
    assert not f(ctx, -1, views, 3, P, L, None, R, None)
    assert not f(ctx, 2, views, -1, P, L, None, R, None)
    assert not f(ctx, 2, views, 3, None, L, None, R, None)
    assert not f(ctx, 2, views, 3, P, None, None, R, None)
    assert not f(ctx, 2, None, 3, P, L, None, R, None)
    assert not f(ctx, 2, views, 3, P, L + 4, None, R, None)           # misaligned labels
    assert f(ctx, 0, views, 3, P, L, None, R, None)
    assert f(ctx, 2, views, 0, P, L, None, R, None)
    assert f(ctx, 0, None, 0, None, None, None, None, None)
    torch.cuda.synchronize()
    assert (lab == 7.0).all().item() and (rng == 7.0).all().item()
    hp = np.array([[C1_LAT + 0.05, C1_LON, 500.]] * 3, np.float64)
    hl = np.full((2, 3, 4), 7.0, np.float32)
    g = lib.horizonator_annotate_batch
    assert not g(ctx, -1, views, 3, hp.ctypes.data, hl.ctypes.data)
    assert not g(ctx, 2, views, -1, hp.ctypes.data, hl.ctypes.data)
    assert not g(ctx, 2, views, 3, None, hl.ctypes.data)
    assert not g(ctx, 2, views, 3, hp.ctypes.data, None)
    assert g(ctx, 0, views, 3, hp.ctypes.data, hl.ctypes.data)
    assert g(ctx, 2, views, 0, hp.ctypes.data, hl.ctypes.data)
    assert (hl == 7.0).all()
    assert h.annotate([], hp).shape == (0, 3) and h.annotate([(C1_LAT, C1_LON, 0., 90.)], []).shape == (1, 0)
    # and a valid call does write
    assert g(ctx, 2, views, 3, hp.ctypes.data, hl.ctypes.data) and not (hl == 7.0).all()


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
        from tools.pois import summits
        h = hz.horizonator(C1_LAT, C1_LON, 800, 200, dir_dems=tiles, render_radius_cells=600)
        views = [(C1_LAT + 0.011 * k, C1_LON - 0.009 * k, 10. * k, 10. * k + 120.) for k in range(-6, 7)]
        pois = summits(h, 400, seed=8)
        want = h.annotate(views, pois)
        got = sharding.annotate_sharded(h, views, pois)
        ok = np.array_equal(got.cpu().numpy().view(np.uint32).reshape(want.shape + (4,)),
                            want.view(np.float32).reshape(want.shape + (4,)).view(np.uint32))
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def test_nccl_sharded_labels_equal_one_gpu(tiles_c1):
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
