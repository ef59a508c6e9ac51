"""Viewsheds without a GPU: the oracle's restatement of R2 (include/horizonator-batch.h) against closed forms and
against brute-force line of sight on the same triangulation, its independence of the thread count, and the sum of
per-rank counts that sharding.viewshed_counts_sharded() does (gloo, as test_sharding.py)."""
import os
import socket

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON
from oracle.binding import Oracle
from oracle.viewshed import ViewshedOracle, eye_at

CURVATURE = (1.0 - 0.13) / (2.0 * 6371000.0)        # horizonator_set_earth_curvature(on, refraction 0.13)
EYES = ["centre", "vertex", "corner sw", "corner ne", "last cell e", "last cell n"]


def _vertex(o, n):
    """the reachable integer cell coordinate (the same along both axes here) nearest the middle of the square"""
    for c in sorted(range(n - 1), key=lambda c: abs(c - n // 2)):
        o.move(*eye_at(o, c, c))
        v = o.viewer()
        if v["viewer_cell_i"] == c and v["viewer_cell_j"] == c:
            return c
    raise AssertionError("no vertex reachable")


def _move(o, where, viewer_z=None):
    """Puts the oracle's eye at one of EYES: the C1 viewpoint, exactly on a vertex, in a corner cell (a quarter of a
    cell in, and the largest reachable coordinates below N - 1), in the last cell of the east and of the north side"""
    n = 2 * o.dem_geometry()["radius_cells"]
    mid, top = (n - 1) / 2 + 0.2, ("below", n - 1)
    if where == "vertex":
        c = _vertex(o, n)
        ci, cj = c, c
    else:
        ci, cj = {"corner sw": (0.25, 0.25), "corner ne": (top, top), "last cell e": (top, mid),
                  "last cell n": (mid, top)}.get(where, (None, None))
    lat, lon = (C1_LAT, C1_LON) if where == "centre" else eye_at(o, ci, cj)
    o.move(lat, lon, viewer_z)
    v = o.viewer()
    if where == "vertex":
        assert v["viewer_cell_i"] == ci and v["viewer_cell_j"] == cj
    elif where != "centre":
        for c, got in ((ci, v["viewer_cell_i"]), (cj, v["viewer_cell_j"])):
            assert (c[1] - 0.05 < got < c[1]) if isinstance(c, tuple) else (c <= got < c + 0.05), (where, v)
    print(where, "eye cell", v["viewer_cell_i"], v["viewer_cell_j"], "z", v["viewer_z"])
    return v


def _metres(o):
    """(north, east) metres of every vertex from the eye, (N, N) each, in double."""
    g, v = o.dem_geometry(), o.viewer()
    n = 2 * g["radius_cells"]
    cell = 6371000.0 * np.pi / 180.0 / g["cells_per_deg"]
    idx = np.arange(n, dtype=np.float64)
    north = (idx - v["viewer_cell_j"]) * cell
    east = (idx - v["viewer_cell_i"]) * cell * v["cos_viewer_lat"]
    return north[:, None] + 0 * east[None, :], east[None, :] + 0 * north[:, None]


def test_flat_ground_flat_earth_sees_everything(tmp_path):
    o = Oracle(C1_LAT, C1_LON, 64, 16, dir_dems=str(tmp_path), render_radius_cells=120, threads=4)
    vs = ViewshedOracle(o, threads=4)
    for dl in ((0.0, 0.0), (0.03, -0.04)):
        o.move(C1_LAT + dl[0], C1_LON + dl[1])
        assert vs.mask().all()


@pytest.mark.parametrize("viewer_z", [None, 0.0])
@pytest.mark.parametrize("where", EYES)
@pytest.mark.parametrize("R", [1, 2, 17, 120])
def test_flat_ground_flat_earth_sees_everything_from_any_eye(tmp_path, R, where, viewer_z):
    """N in {2, 4, 34, 240}, eyes on a vertex and in the outermost cells.  With the eye on the ground (viewer_z 0)
    every slope is 0 and every comparison with the running maximum a tie, which counts as visible."""
    o = Oracle(C1_LAT, C1_LON, 64, 16, dir_dems=str(tmp_path), render_radius_cells=R, threads=4)
    vs = ViewshedOracle(o, threads=4)
    v = _move(o, where, viewer_z)
    assert v["viewer_z"] == (1.0 if viewer_z is None else 0.0)
    words = vs.words()
    n = 2 * R
    assert vs.mask().all()
    assert not (words[:, -1] >> np.uint32(n % 32)).any() if n % 32 else True


def _assert_geometric_horizon(o):
    """flat ground, curvature on: the auto eye (1 m up) sees everything inside the geometric horizon, nothing beyond"""
    vz = o.viewer()["viewer_z"]
    assert vz == 1.0                                       # auto eye: the ground (0) + 1 m
    m = ViewshedOracle(o, threads=4).mask(curvature=CURVATURE)
    north, east = _metres(o)
    d = np.hypot(north, east)
    horizon = np.sqrt(vz / CURVATURE)                      # slope -vz/d - c*d peaks there
    slack = np.hypot(92.7, 92.7)                           # one cell
    assert m[d < horizon - slack].all()
    assert not m[d > horizon + slack].any()
    return m, d, horizon


def test_flat_ground_with_curvature_ends_at_the_geometric_horizon(tmp_path):
    o = Oracle(C1_LAT, C1_LON, 64, 16, dir_dems=str(tmp_path), render_radius_cells=100, threads=4)
    m, d, horizon = _assert_geometric_horizon(o)
    assert 40 * 75 < horizon < 0.6 * d.max()
    assert 0.0 < m.mean() < 0.5


@pytest.mark.parametrize("where", EYES)
@pytest.mark.parametrize("R", [1, 2, 17, 100])
def test_flat_ground_with_curvature_ends_at_the_geometric_horizon_from_any_eye(tmp_path, R, where):
    """The 1 m eye's geometric horizon is 3.8 km away: beyond the tiny squares but for the far corner of N = 34"""
    o = Oracle(C1_LAT, C1_LON, 64, 16, dir_dems=str(tmp_path), render_radius_cells=R, threads=4)
    _move(o, where)
    m, d, horizon = _assert_geometric_horizon(o)
    if R == 100:
        assert 40 * 75 < horizon < 0.6 * d.max()
        assert 0.0 < m.mean() < 0.5


def _ridge_tiles(directory, col=20, height=50):
    """Zero tiles around the C1 eye with one north-south wall `height` m high on column `col` of the W117 tiles."""
    for lat in (34, 35):
        for lon in (-118, -117):
            z = np.zeros((1201, 1201), ">i2")
            if lon == -117:
                z[:, col] = height
            z.tofile(os.path.join(directory, "N%02dW%03d.hgt" % (lat, -lon)))
    return directory


def _assert_ridge_shadow(o, diagonal):
    """The closed-form shadow of _ridge_tiles()'s wall from o's eye; diagonal: whether vertices exactly on a diagonal
    through the eye count as decided by column-stepping rays alone (from an eye on a vertex a row-stepping ray ends
    on the same corner and decides them too)"""
    mos = o.mosaic()
    walls = np.where((mos == 50).all(axis=0))[0]
    assert len(walls) == 1 and (mos[:, np.arange(mos.shape[1]) != walls[0]] == 0).all()
    ic = int(walls[0])
    v = o.viewer()
    vci, vcj = v["viewer_cell_i"], v["viewer_cell_j"]
    assert 10 < ic - vci < 40
    m = ViewshedOracle(o, threads=4).mask()
    n = m.shape[0]
    jj, ii = np.mgrid[0:n, 0:n].astype(np.float64)
    di, dj = ii - vci, jj - vcj
    column_rays = ((np.abs(dj) <= np.abs(di)) if diagonal else (np.abs(dj) < np.abs(di))) & (di > 1)
    expect = ~((ii > ic) & (di < 2 * (ic - vci)))
    bad = column_rays & (m != expect)
    slack = (np.abs(di - (ic - vci)) <= 1) | (np.abs(di - 2 * (ic - vci)) <= 1)
    assert not (bad & ~slack).any(), np.argwhere(bad & ~slack)[:10]
    shadow = column_rays & (ii > ic + 1) & (di < 2 * (ic - vci) - 1)
    assert shadow.sum() > 500 and not m[shadow].any()


def test_straight_ridge_casts_the_closed_form_shadow(tmp_path):
    """Eye 100 m up, a 50 m wall at column ic east of it: behind the wall the ground is hidden from the wall out to
    twice the wall's distance (the slope to the ground, -100/d, equals the wall's, -50/d_wall, at d = 2 d_wall).
    Checked on the vertices whose rays step over columns (they sample the wall at its full height); one cell of slack."""
    d = _ridge_tiles(str(tmp_path))
    o = Oracle(C1_LAT, C1_LON, 64, 16, dir_dems=d, render_radius_cells=100, viewer_z=100.0, threads=4)
    _assert_ridge_shadow(o, diagonal=True)


RIDGE_EYES = {"vertex": (99, 99), "grid line": (99, 60.4), "corner sw": (99.5, 0.25),
              "last cell n": (99.5, ("below", 199))}


@pytest.mark.parametrize("where", RIDGE_EYES)
def test_straight_ridge_casts_the_closed_form_shadow_from_edge_eyes(tmp_path, where):
    """The same wall from eyes on a vertex (column 99 is the W117 tile's west edge), on a vertical grid line, near the
    south-west corner and in the last cell of the north side"""
    d = _ridge_tiles(str(tmp_path))
    o = Oracle(C1_LAT, C1_LON, 64, 16, dir_dems=d, render_radius_cells=100, viewer_z=100.0, threads=4)
    o.move(*eye_at(o, *RIDGE_EYES[where]), viewer_z=100.0)
    v = o.viewer()
    print(where, "eye cell", v["viewer_cell_i"], v["viewer_cell_j"])
    if where in ("vertex", "grid line"):
        assert v["viewer_cell_i"] == 99 and v["viewer_cell_j"].is_integer() == (where == "vertex")
    _assert_ridge_shadow(o, diagonal=where != "vertex")


@pytest.mark.parametrize("dlat,dlon", [(0.0, 0.0), (0.03, -0.02), (-0.04, 0.05)])
def test_r2_against_exact_line_of_sight(tiles_c1, dlat, dlon):
    """R2 approximates line of sight: at most 3 % of the vertices disagree with brute-force line of sight on the same
    triangulation, at most 0.5 % are visible vertices that R2 calls hidden."""
    o = Oracle(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_c1, render_radius_cells=150, threads=os.cpu_count() or 1)
    o.move(C1_LAT + dlat, C1_LON + dlon)
    vs = ViewshedOracle(o)
    r2, exact = vs.mask(), vs.mask(exact=True)
    disagree, missed = (r2 != exact).mean(), (exact & ~r2).mean()
    print("R2 vs exact at", (dlat, dlon), "visible %.4f / %.4f, disagree %.4f, missed %.4f"
          % (r2.mean(), exact.mean(), disagree, missed))
    assert exact.mean() > 0.001
    assert disagree <= 0.03 and missed <= 0.005


def test_mask_does_not_depend_on_the_thread_count(tiles_c1):
    o = Oracle(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_c1, render_radius_cells=300, threads=1)
    o.move(C1_LAT - 0.02, C1_LON + 0.01)
    vs = ViewshedOracle(o, threads=1)
    one = vs.words(1.7)
    for t in (2, 7, os.cpu_count() or 1):
        vs.threads = t
        assert np.array_equal(vs.words(1.7), one)


def test_eye_outside_the_square_is_refused(tiles_c1):
    o = Oracle(C1_LAT, C1_LON, 64, 16, dir_dems=tiles_c1, render_radius_cells=50, threads=1)
    o.move(C1_LAT + 0.2, C1_LON)
    with pytest.raises(ValueError):
        ViewshedOracle(o).mask()


# ---------------------------------------------------------------------------------------------- sharded counts

def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _counts(rank, n=37):
    return np.random.default_rng(rank).integers(0, 100, (n, n)).astype(np.int32)


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    from horizonator_b200 import sharding
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        total = sum(_counts(r) for r in range(world))
        c = sharding.reduce_counts(torch.from_numpy(_counts(rank)))
        ok = np.array_equal(c.numpy(), total)
        c = sharding.reduce_counts(torch.from_numpy(_counts(rank)), root=1)
        if rank == 1:
            ok = ok and np.array_equal(c.numpy(), total)
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_sharded_counts_sum(world):
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


def test_single_process_counts_need_no_process_group():
    import torch
    from horizonator_b200 import sharding
    c = torch.from_numpy(_counts(0))
    assert sharding.reduce_counts(c) is c
