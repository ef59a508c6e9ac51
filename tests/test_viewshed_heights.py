"""Viewshed heights without a GPU: the oracle's restatement (vs_oracle_r2_heights, include/horizonator-batch.h) against
closed forms -- flat ground, the curvature horizon, the shadow of a straight wall -- against the oracle's own masks,
its independence of the thread count, and the minimum over ranks that sharding.viewshed_least_height_sharded() takes
(gloo, as test_sharding.py)."""
import os
import socket

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON
from oracle.binding import Oracle
from oracle.viewshed import ViewshedOracle, eye_at
from oracle.viewshed_heights import r2_heights

CURVATURE = (1.0 - 0.13) / (2.0 * 6371000.0)        # horizonator_set_earth_curvature(on, refraction 0.13)
CELL_N = 6371000.0 * np.pi / 180.0 / 1200.0           # metres per SRTM3 cell, north


def _vertex(o, n):
    """the reachable integer cell coordinate (the same along both axes) nearest the middle of the square"""
    for c in sorted(range(n - 1), key=lambda c: abs(c - n // 2)):
        o.move(*eye_at(o, c, c), o.fixed_z)
        v = o.viewer()
        if v["viewer_cell_i"] == c and v["viewer_cell_j"] == c:
            return c
    raise AssertionError("no vertex reachable")


def _eye(o, where):
    """Puts o's eye at the C1 viewpoint, exactly on a vertex, or in a corner or side's outermost cell; returns it"""
    n = 2 * o.dem_geometry()["radius_cells"]
    top, mid = ("below", n - 1), (n - 1) / 2 + 0.2
    if where == "vertex":
        _vertex(o, n)
        return o.viewer()
    cells = {"corner sw": (0.25, 0.25), "corner ne": (top, top), "last cell e": (top, mid), "last cell n": (mid, top)}
    lat, lon = (C1_LAT, C1_LON) if where == "centre" else eye_at(o, *cells[where])
    o.move(lat, lon, o.fixed_z)
    return o.viewer()


def _metres(o):
    """(north, east) metres of every vertex from the eye, (N, N) each, in double"""
    g, v = o.dem_geometry(), o.viewer()
    n = 2 * g["radius_cells"]
    cell = 6371000.0 * np.pi / 180.0 / g["cells_per_deg"]
    idx = np.arange(n, dtype=np.float64)
    north = (idx[:, None] - v["viewer_cell_j"]) * cell + 0 * idx[None, :]
    east = (idx[None, :] - v["viewer_cell_i"]) * cell * v["cos_viewer_lat"] + 0 * idx[:, None]
    return north, east


def _oracle(tiles, R, viewer_z=None, threads=4):
    o = Oracle(C1_LAT, C1_LON, 64, 16, dir_dems=tiles, render_radius_cells=R, viewer_z=viewer_z, threads=threads)
    o.fixed_z = viewer_z                                 # None: automatic, 1 m over the ground
    return o


def _assert_valid(h):
    """every height >= +0 (never -0) or +inf, never NaN"""
    assert h.dtype == np.float32
    assert not np.isnan(h).any() and (h >= 0).all() and not np.signbit(h).any()


@pytest.mark.parametrize("viewer_z", [None, 0.0, 250.0])
@pytest.mark.parametrize("where", ["centre", "vertex", "corner sw", "corner ne", "last cell e", "last cell n"])
@pytest.mark.parametrize("R", [1, 17, 120])
def test_flat_ground_flat_earth_needs_no_height(tmp_path, R, where, viewer_z):
    """No tiles: from any eye the ground slopes away monotonically (or is level with an eye on it), so every vertex is
    seen at the ground, +0 exactly"""
    o = _oracle(str(tmp_path), R, viewer_z)
    v = _eye(o, where)
    h = r2_heights(ViewshedOracle(o, threads=4))
    print(where, "eye cell", v["viewer_cell_i"], v["viewer_cell_j"], "z", v["viewer_z"])
    _assert_valid(h)
    assert (h == 0).all()


@pytest.mark.parametrize("where", ["centre", "vertex", "corner sw", "last cell n"])
def test_flat_ground_with_curvature_closed_form(tmp_path, where):
    """Eye 1 m over flat ground, curvature c: the ground's slope -1/d - c d peaks at the geometric horizon
    d_h = 1/sqrt(c) (3.83 km), at -2 sqrt(c), so a point at distance D beyond it is seen from the height
    (sqrt(c) D - 1)^2 up.  The rays' largest slope is at most the peak, so R2's heights are at most the closed form; the
    step nearest d_h is at most half a step away, where the slope is below the peak by at most c^1.5 (step / 2)^2, so
    they are at least the closed form minus D times that.  Inside the horizon every height is +0."""
    o = _oracle(str(tmp_path), 100)
    v = _eye(o, where)
    assert v["viewer_z"] == 1.0
    h = r2_heights(ViewshedOracle(o, threads=4), curvature=CURVATURE)
    _assert_valid(h)
    north, east = _metres(o)
    D = np.hypot(north, east)
    dh = 1.0 / np.sqrt(CURVATURE)
    step = np.hypot(CELL_N, CELL_N)                      # the longest step of a ray, along a diagonal
    closed = (np.sqrt(CURVATURE) * D - 1.0) ** 2
    rounding = 1e-5 * (1.0 + CURVATURE * D ** 2)         # a few float ulps of the terms smax * D and A
    inside, beyond = D < dh - step, D > dh + 2 * step
    assert inside.sum() > 1000 and beyond.sum() > 1000
    assert (h[inside] == 0).all(), np.argwhere(inside & (h != 0))[:5]
    assert np.isfinite(h).all()
    over = h - closed
    assert (over[beyond] <= rounding[beyond]).all(), over[beyond].max()
    under = closed - h
    bound = D * CURVATURE ** 1.5 * (step / 2) ** 2 + rounding
    assert (under[beyond] <= bound[beyond]).all(), (under - bound)[beyond].max()
    print(where, "beyond the horizon: closed form minus heights in [%.2e, %.2e] m, bound %.2e m"
          % (under[beyond].min(), under[beyond].max(), bound[beyond].max()))


def _ridge_tiles(directory, col=20, height=50):
    """Zero tiles around the C1 eye with one north-south wall `height` m high on column `col` of the W117 tiles."""
    for lat in (34, 35):
        for lon in (-118, -117):
            z = np.zeros((1201, 1201), ">i2")
            if lon == -117:
                z[:, col] = height
            z.tofile(os.path.join(directory, "N%02dW%03d.hgt" % (lat, -lon)))
    return directory


@pytest.mark.parametrize("where", ["centre", "vertex"])
def test_straight_wall_closed_form(tmp_path, where):
    """Eye 100 m up, a 50 m wall at column ic east of it.  A column-stepping ray that crosses the wall at distance
    d_w keeps the wall's slope -50 / d_w as its largest until the ground's -100 / d overtakes it at d = 2 d_w, so a
    vertex behind the wall at distance D is seen from 100 - 50 D / d_w up, and from the ground (+0) from twice the
    wall's distance on.  Along a ray d_w / d = (ic - eye_i) / (i - eye_i); the vertex is up to half a row off the ray,
    so its D differs from the ray's own distance by at most half a cell north: that is the tolerance.  Checked on
    vertices more than a cell off the diagonals, which only column-stepping rays decide."""
    d = _ridge_tiles(str(tmp_path))
    o = _oracle(d, 100, viewer_z=100.0)
    v = _eye(o, where)
    mos = o.mosaic()
    walls = np.where((mos == 50).all(axis=0))[0]
    assert len(walls) == 1
    ic = int(walls[0])
    vci, vcj = v["viewer_cell_i"], v["viewer_cell_j"]
    assert 10 < ic - vci < 40
    h = r2_heights(ViewshedOracle(o, threads=4))
    _assert_valid(h)
    n = h.shape[0]
    jj, ii = np.mgrid[0:n, 0:n].astype(np.float64)
    di, dj = ii - vci, jj - vcj
    north, east = _metres(o)
    D = np.hypot(north, east)
    cols = (np.abs(dj) < np.abs(di) - 1) & (di > 1)
    w = ic - vci
    behind = cols & (ii > ic) & (di < 2 * w - 1)
    expect = 100.0 - 50.0 * di / w
    tol = 50.0 * di / w * 0.5 * CELL_N / (D - 0.5 * CELL_N) + 1e-3
    assert behind.sum() > 500
    err = np.abs(h - expect)
    assert (err[behind] <= tol[behind]).all(), np.argwhere(behind & (err > tol))[:5]
    assert (h[behind] > 0).all()
    # in front of the wall, on it, and from twice its distance on: the ground is seen
    assert (h[cols & ((ii <= ic) | (di > 2 * w + 1))] == 0).all()
    print(where, "wall at %.2f cells: %d vertices behind it, largest error %.3f m (tolerance there %.3f m)"
          % (w, behind.sum(), err[behind].max(), tol[behind][np.argmax(err[behind])]))


def test_heights_do_not_depend_on_the_thread_count(tiles_c1):
    o = _oracle(tiles_c1, 300, threads=1)
    o.move(C1_LAT - 0.02, C1_LON + 0.01)
    vs = ViewshedOracle(o, threads=1)
    for c in (0.0, CURVATURE):
        vs.threads = 1
        one = r2_heights(vs, curvature=c)
        _assert_valid(one)
        for t in (2, 7, os.cpu_count() or 1):
            vs.threads = t
            assert np.array_equal(r2_heights(vs, curvature=c).view(np.uint32), one.view(np.uint32)), (c, t)


@pytest.mark.parametrize("curvature", [0.0, CURVATURE])
@pytest.mark.parametrize("where", ["centre", "vertex", "corner ne", "last cell e"])
def test_heights_agree_with_the_masks(tiles_c1, where, curvature):
    """isfinite(heights) is the mask at t = 1e30 exactly; the mask at t is heights <= t but where t is within rounding
    of a step's terms (|height - t| < 0.01 m)"""
    o = _oracle(tiles_c1, 300, threads=os.cpu_count() or 1)
    v = _eye(o, where)
    vs = ViewshedOracle(o)
    h = r2_heights(vs, curvature=curvature)
    _assert_valid(h)
    assert np.array_equal(np.isfinite(h), vs.mask(1e30, curvature=curvature))
    print(where, "eye cell", v["viewer_cell_i"], v["viewer_cell_j"], "+inf vertices:", int(np.isinf(h).sum()))
    seen = []
    for t in (0.0, 1.7, 10.0, 250.0):
        m = vs.mask(t, curvature=curvature)
        seen.append(m.mean())
        near = np.abs(h - np.float32(t)) < 0.01
        differ = m != (h <= np.float32(t))
        print("  t = %g m: %d vertices within 0.01 m of t, %d of them differ; seen %.4f"
              % (t, near.sum(), (differ & near).sum(), m.mean()))
        assert not (differ & ~near).any(), np.argwhere(differ & ~near)[:5]
    assert 0 < seen[0] < seen[-1] < 0.999


def test_eye_outside_the_square_is_refused(tiles_c1):
    o = _oracle(tiles_c1, 50, threads=1)
    o.move(C1_LAT + 0.2, C1_LON)
    with pytest.raises(ValueError):
        r2_heights(ViewshedOracle(o))


# ---------------------------------------------------------------------------------------------- sharded least

def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _least(rank, n=37):
    """a rank's least heights: non-negative floats, +0 and +inf among them"""
    rs = np.random.default_rng(rank)
    x = rs.exponential(30.0, (n, n)).astype(np.float32)
    x[rs.random((n, n)) < 0.2] = np.inf
    x[rs.random((n, n)) < 0.1] = 0.0
    return x


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    from horizonator_b200 import sharding
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        want = np.minimum.reduce([_least(r) for r in range(world)])
        x = sharding.reduce_least(torch.from_numpy(_least(rank)))
        ok = np.array_equal(x.numpy().view(np.uint32), want.view(np.uint32))
        x = sharding.reduce_least(torch.from_numpy(_least(rank)), root=1)
        if rank == 1:
            ok = ok and np.array_equal(x.numpy().view(np.uint32), want.view(np.uint32))
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_sharded_least_is_the_minimum(world):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    got = sorted(q.get(timeout=5) for _ in range(world))
    assert got == [(r, True) for r in range(world)]


def test_single_process_least_needs_no_process_group():
    import torch
    from horizonator_b200 import sharding
    x = torch.from_numpy(_least(0))
    assert sharding.reduce_least(x) is x
