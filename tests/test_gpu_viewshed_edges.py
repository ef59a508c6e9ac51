"""Viewsheds on the GPU against the oracle (vs_oracle_r2) bit for bit, whole uint32 words with their unused tail bits,
where k_viewshed's hand-built parts can go wrong: every mask width and warp padding from N = 2 up, eyes exactly on grid
lines and vertices and in the outermost cells, ties of the running maximum on flat ground, explicit eye heights and
extreme target heights, missing tiles and voids, earth curvature, chunks of 64 views with the counts and the scratch,
the host-memory call's += on the caller's counts, side streams, and viewsheds between renders and curvature changes.
Run on the B200 box: pytest -m gpu."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON
from oracle import vertex
from oracle.viewshed import ViewshedOracle, eye_at, unpack_mask

pytestmark = pytest.mark.gpu

POISON = 0x5A5A5A5A
C2_LAT, C2_LON = 34.0 + 1.0 / 7200.0, -117.0 + 1.0 / 7200.0


def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test running without a CUDA device"
    return torch


class Pair:
    """A product context and an oracle over the same tiles and square, both made at (lat, lon)."""

    def __init__(self, hz, tiles, R, srtm1, lat, lon):
        from oracle.binding import Oracle
        kw = dict(render_radius_m=150000.) if R is None else dict(render_radius_cells=R)
        self.hz = hz
        self.h = hz.horizonator(lat, lon, 64, 16, SRTM1=srtm1, dir_dems=tiles, **kw)
        self.o = Oracle(lat, lon, 64, 16, SRTM1=srtm1, dir_dems=tiles, threads=os.cpu_count() or 1, **kw)
        self.vs = ViewshedOracle(self.o)
        self.N = self.h.size
        assert self.N == self.vs.heights.shape[0]
        self.w32 = (self.N + 31) // 32

    def view(self, ci, cj, viewer_z=None):
        """A view whose eye is at cell coordinates (ci, cj) as eye_at() places it, checked on the oracle: a coordinate
        is a rounded product of the float32 angle, so it lands within a few hundredths of a cell at or above the one
        asked for, or below ("below", t)."""
        lat, lon = eye_at(self.o, ci, cj)
        self.o.move(lat, lon)
        v = self.o.viewer()
        for c, got in ((ci, v["viewer_cell_i"]), (cj, v["viewer_cell_j"])):
            if isinstance(c, tuple):
                assert c[1] - 0.05 < got < c[1], (ci, cj, v)
            else:
                assert c <= got < c + 0.05, (ci, cj, v)
        return (lat, lon) if viewer_z is None else (lat, lon, 0., 0., float(viewer_z))

    def integer(self, near, axis):
        """The reachable integer cell coordinate (axis 0: i, 1: j) nearest `near`: only some integers are"""
        for c in sorted(range(1, self.N - 1), key=lambda c: abs(c - near)):
            lat, lon = eye_at(self.o, *((c, 1.5) if axis == 0 else (1.5, c)))
            self.o.move(lat, lon)
            if self.o.viewer()["viewer_cell_" + "ij"[axis]] == c:
                return c
        raise AssertionError("no integer cell coordinate reachable near %g" % near)

    def on_vertex(self, near_i, near_j, viewer_z=None):
        """A view whose eye is exactly on the reachable vertex nearest (near_i, near_j)"""
        return self.view(self.integer(near_i, 0), self.integer(near_j, 1), viewer_z)

    def oracle_words(self, view, th=0., curvature=0.):
        """The oracle's mask of one view, and its eye"""
        self.o.move(view[0], view[1], view[4] if len(view) > 4 else None)
        return self.vs.words(th, curvature=curvature), self.o.viewer()

    def device(self, views, th=0., counts=None, stream=None):
        """One horizonator_viewshed_device call into masks poisoned with POISON: (n, N, W32) uint32 on the host"""
        torch = _torch()
        d = torch.full((len(views), self.N, self.w32), POISON, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()            # the context's own stream does not wait for torch's fills
        ok = self.hz.lib.horizonator_viewshed_device(
            C.byref(self.h.context), len(views), self.h._eyes(views), float(th), d.data_ptr(),
            counts.data_ptr() if counts is not None else None, stream)
        assert ok, "horizonator_viewshed_device refused the views"
        torch.cuda.synchronize()
        return d.cpu().numpy().view(np.uint32)


def _side(i, j, vci, vcj, N):
    """Which side of the square the ray through vertex (i, j) ends on"""
    di, dj = i - float(vci), j - float(vcj)
    ti = ((N - 1 - float(vci)) / di if di > 0 else -float(vci) / di) if di else np.inf
    tj = ((N - 1 - float(vcj)) / dj if dj > 0 else -float(vcj) / dj) if dj else np.inf
    if ti <= tj:
        return "right column" if di > 0 else "left column"
    return "top row" if dj > 0 else "bottom row"


def assert_same(got, want, v, N, what=""):
    """Whole words equal, tail bits 0; on a difference: how many bits, where, the eye and the sides of the rays"""
    tail = np.uint32((1 << (N % 32)) - 1) if N % 32 else np.uint32(0xFFFFFFFF)
    assert not (got[:, -1] & ~tail).any(), "%s: unused tail bits set by the kernel" % what
    assert not (want[:, -1] & ~tail).any(), "%s: unused tail bits set by the oracle" % what
    if np.array_equal(got, want):
        return
    nbits = int(np.unpackbits((got ^ want).view(np.uint8)).sum())
    jj, ii = np.nonzero(unpack_mask(got) != unpack_mask(want))
    g = unpack_mask(got)
    first = ["(%d, %d) kernel %d, %s" % (i, j, g[j, i], _side(i, j, v["viewer_cell_i"], v["viewer_cell_j"], N))
             for i, j in zip(ii[:6], jj[:6])]
    raise AssertionError("%s: %d bits differ, N = %d, eye cell (%r, %r), z %r; first %s"
                         % (what, nbits, N, v["viewer_cell_i"], v["viewer_cell_j"], v["viewer_z"], "; ".join(first)))


def check(pair, views, th=0., curvature=0., what="", counts=None, stream=None):
    """Kernel against oracle for every view of one call; returns the kernel's words and the oracle's masks"""
    got = pair.device(views, th, counts, stream)
    masks = []
    for k, view in enumerate(views):
        want, v = pair.oracle_words(view, th, curvature)
        print("%s view %d: eye cell (%r, %r), z %r, visible %.5f" % (what, k, v["viewer_cell_i"], v["viewer_cell_j"],
                                                                     v["viewer_z"], unpack_mask(want).mean()))
        assert_same(got[k], want, v, pair.N, "%s view %d" % (what, k))
        masks.append(unpack_mask(want))
    return got, np.array(masks)


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


# ---------------------------------------------------------------------------------------------- mask widths

@pytest.mark.parametrize("where", ["centre", "corner"])
@pytest.mark.parametrize("R", [1, 2, 3, 15, 16, 17, 31, 33, 47, 300])
def test_every_mask_width(pairs, tiles_c1, R, where):
    """N = 2R in {2, 4, 6, 30, 32, 34, 62, 66, 94, 600}: N % 32 in {0, 2, 4, 6, 24, 30}, N - 2 on both sides of
    multiples of 32 (the column sides' warps), down to a square without column rays (N = 2)"""
    p = pairs(tiles_c1, R)
    N = p.N
    assert N == 2 * R
    view = (C1_LAT, C1_LON) if where == "centre" else p.view(("below", N - 1), 0.3)
    _, m = check(p, [view], what="N %d %s" % (N, where))
    if N >= 66:
        assert 0.001 < m.mean() < 0.999, m.mean()


# ---------------------------------------------------------------------------------------------- eye placements

# eyes on grid lines and vertices, in the outermost cells, at the extreme reachable coordinates: name -> view of a
# Pair p whose square has R = N / 2
PLACEMENTS = {
    "vertex": lambda p, R, N: p.on_vertex(R + 20, R - 30),
    "vertical line": lambda p, R, N: p.view(p.integer(R + 20, 0), R + 0.37),
    "horizontal line": lambda p, R, N: p.view(R - 0.41, p.integer(R - 30, 1)),
    "corner sw": lambda p, R, N: p.view(0.5, 0.5),
    "corner se": lambda p, R, N: p.view(N - 1.5, 0.5),
    "corner nw": lambda p, R, N: p.view(0.5, N - 1.5),
    "corner ne": lambda p, R, N: p.view(N - 1.5, N - 1.5),
    "side w": lambda p, R, N: p.view(0.5, R + 0.3),
    "side e": lambda p, R, N: p.view(N - 1.5, R + 0.3),
    "side s": lambda p, R, N: p.view(R + 0.3, 0.5),
    "side n": lambda p, R, N: p.view(R + 0.3, N - 1.5),
    "lowest": lambda p, R, N: p.view(0.0, 0.0),
    "highest": lambda p, R, N: p.view(("below", N - 1), ("below", N - 1)),
    "highest i": lambda p, R, N: p.view(("below", N - 1), R + 0.3),
    "highest j": lambda p, R, N: p.view(R - 0.3, ("below", N - 1)),
}


def _place(p, name):
    return PLACEMENTS[name](p, p.N // 2, p.N)


@pytest.mark.parametrize("name", PLACEMENTS)
@pytest.mark.parametrize("R", [300, 1200])
def test_eye_placements(pairs, tiles_c1, R, name):
    p = pairs(tiles_c1, R)
    view = _place(p, name)
    _, v = p.oracle_words(view)
    ci, cj = v["viewer_cell_i"], v["viewer_cell_j"]
    if name == "vertex":
        assert ci.is_integer() and cj.is_integer()
    elif name == "vertical line":
        assert ci.is_integer() and not cj.is_integer()
    elif name == "horizontal line":
        assert cj.is_integer() and not ci.is_integer()
    elif name == "lowest":
        assert 0 <= ci < 0.01 and 0 <= cj < 0.01
    elif name.startswith("highest"):
        assert max(ci, cj) > p.N - 1.05
    check(p, [view], what="R %d %s" % (R, name))
    check(p, [view], 1.7, what="R %d %s, target 1.7 m" % (R, name))
    if name in ("vertex", "vertical line", "horizontal line"):
        # an eye just under the ground: the surface on the eye's own grid line is above it (a slope of +inf there),
        # so a ray that also stepped onto that line would hide everything beyond
        i0, j0 = int(np.floor(ci)), int(np.floor(cj))
        z = float(p.vs.heights[j0:j0 + 2, i0:i0 + 2].min()) - 0.25
        check(p, [view[:2] + (0., 0., z)], what="R %d %s, eye %g m" % (R, name, z))


def test_eyes_at_the_square_edge_are_refused_by_both(hz, pairs, tiles_c1):
    """The next float32 angle above the highest accepted eye puts the eye on the square's last vertex line: both the
    kernel's host side and the oracle refuse it, and the call writes nothing"""
    torch = _torch()
    p = pairs(tiles_c1, 300)
    N = p.N
    for ci, cj in ((("below", N - 1), 300.3), (300.3, ("below", N - 1))):
        lat, lon = p.view(ci, cj)
        up = lambda x: float(np.nextafter(np.float32(x), np.float32(np.inf)))
        bad = (lat, up(lon)) if isinstance(ci, tuple) else (up(lat), lon)
        p.o.move(*bad)
        v = p.o.viewer()
        assert max(v["viewer_cell_i"], v["viewer_cell_j"]) == N - 1, v
        with pytest.raises(ValueError):
            p.vs.words()
        masks = torch.full((2, N, p.w32), POISON, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        assert not hz.lib.horizonator_viewshed_device(C.byref(p.h.context), 2, p.h._eyes([(lat, lon), bad]), 0.,
                                                      masks.data_ptr(), None, None)
        torch.cuda.synchronize()
        assert (masks == POISON).all().item()


# ---------------------------------------------------------------------------------------------- heights

@pytest.mark.parametrize("R", [300, 1200])
def test_explicit_eye_heights(pairs, tiles_c1, R):
    """viewer_z = 0 given explicitly (not the automatic eye), below most of the terrain, and 9000 m"""
    p = pairs(tiles_c1, R)
    low = float(np.percentile(p.vs.heights, 10))
    views = [p.view(R - 0.3, R + 0.2, z) for z in (0., low, 9000.)] + [p.on_vertex(R + 20, R - 30, 0.)]
    for th in (0., 1.7):
        _, m = check(p, views, th, what="R %d explicit z, target %g" % (R, th))
        # under the terrain the eye sees the four vertices around it and little else; 9000 m up, most of the square
        assert m[0].mean() <= m[1].mean() < m[2].mean() and m[2].mean() > 0.5


@pytest.mark.parametrize("th", [-50., 0., 1.7, 250., 1e4])
def test_target_heights(pairs, tiles_c1, th):
    p = pairs(tiles_c1, 1200)
    views = [(C1_LAT, C1_LON), p.view(0.5, 2398.5), p.on_vertex(1220, 1170)]
    _, m = check(p, views, th, what="target %g" % th)
    if th == 1e4:
        assert m.mean() > 0.5


@pytest.mark.parametrize("R", [2, 17, 300])
def test_flat_ground_ties_everywhere(pairs, tiles_flat, R):
    """No tiles, eye at height 0: every slope is 0, every comparison of the running maximum a tie, and every vertex
    visible; with an automatic eye (1 m up) too"""
    p = pairs(tiles_flat, R)
    N = p.N
    assert not p.vs.heights.any()
    views = [p.view(R - 0.3, R + 0.2, 0.), p.view(0.5, ("below", N - 1), 0.), p.view(0.0, 0.0, 0.),
             p.view(R - 0.3, R + 0.2)]
    if R > 2:
        views.append(p.on_vertex(R + 5, R - 7, 0.))
    _, m = check(p, views, what="flat R %d" % R)
    assert m.all()


# ---------------------------------------------------------------------------------------------- terrain

@pytest.mark.parametrize("R", [300, 1200])
def test_missing_and_empty_tiles(pairs, tiles_holes, R):
    p = pairs(tiles_holes, R)
    assert (p.vs.heights == 0).mean() > 0.2
    views = [(C1_LAT, C1_LON), p.view(R + 0.3, R - 0.6), p.view(0.5, 0.5), p.view(("below", p.N - 1), ("below", p.N - 1))]
    check(p, views, 1.7, what="holes R %d" % R)


def test_voids_of_the_synthetic_tiles(pairs, tiles_c1):
    """C1's voids read as 0: eyes next to them"""
    p = pairs(tiles_c1, 1200)
    jj, ii = np.nonzero(p.vs.heights == 0)
    assert len(ii) > 0
    k = np.argsort(np.hypot(ii - 1200, jj - 1200))[0]
    i, j = int(ii[k]), int(jj[k])
    views = [p.view(min(max(i + di, 0.5), 2398.5), min(max(j + dj, 0.5), 2398.5)) for di, dj in ((1.5, 0.5), (-3.5, -2.5))]
    check(p, views, 1.7, what="void at (%d, %d)" % (i, j))


def test_c2_corner_tile_and_last_cell(pairs, tiles_c2):
    """C2 (SRTM1, N = 11716, N % 32 = 4): the eye in the middle of the mesh's south-west tile, and one in the last
    cell of the east side; flat earth and curvature (refraction 0.13)"""
    p = pairs(tiles_c2, None, True)
    assert p.N == 11716
    t = vertex.TILE_CELLS // 2 + 0.5
    views = [p.view(t, t), p.view(("below", p.N - 1), p.N // 2 + 0.3)]
    check(p, views, what="C2")
    try:
        p.h.set_earth_curvature(True, 0.13)
        check(p, views[:1], curvature=vertex.curvature(True, 0.13), what="C2 curved")
    finally:
        p.h.set_earth_curvature(False)


# ---------------------------------------------------------------------------------------------- curvature

REFRACTIONS = [0., 0.13, float(np.nextafter(np.float32(1.0), np.float32(0.0)))]


@pytest.mark.parametrize("refraction", REFRACTIONS)
def test_curvature(pairs, tiles_c1, refraction):
    """set_earth_curvature(True, r) against the oracle given vertex.curvature(True, r).  Refraction is accepted in
    [0, 1): the largest float below 1 leaves a coefficient of a few 1e-15 with the mode on; 1 itself is refused."""
    p = pairs(tiles_c1, 1200)
    views = [(C1_LAT, C1_LON), p.on_vertex(1220, 1170), p.view(0.5, 2398.5)]
    try:
        p.h.set_earth_curvature(True, refraction)
        c = vertex.curvature(True, refraction)
        assert c > 0
        for th in (0., 1.7):
            check(p, views, th, curvature=c, what="refraction %g, target %g" % (refraction, th))
    finally:
        p.h.set_earth_curvature(False)
    with pytest.raises(RuntimeError):
        p.h.set_earth_curvature(True, 1.0)


# ---------------------------------------------------------------------------------------------- batches, host side

def _mixed_views(p):
    """129 views: two whole chunks of 64 and one more, eyes and heights from the cases above"""
    N, R = p.N, p.N // 2
    base = [_place(p, name) for name in PLACEMENTS]
    rs = np.random.default_rng(11)
    views = []
    for k in range(129):
        v = base[k % len(base)][:2]
        z = (-1., 0., 250., 9000.)[k % 4] if k % 3 else float(rs.uniform(0., 1500.))
        if k % 7 == 0:
            v = p.view(float(rs.uniform(0.0, N - 1.01)), float(rs.uniform(0.0, N - 1.01)))[:2]
        views.append(v + (0., 0., z))
    return views


def test_chunks_counts_and_the_host_call(hz, pairs, tiles_c1):
    torch = _torch()
    p = pairs(tiles_c1, 300)
    N = p.N
    views = _mixed_views(p)
    counts = torch.zeros((N, N), dtype=torch.int32, device="cuda")
    got, m = check(p, views, 1.7, what="batch of 129", counts=counts)
    want = m.sum(axis=0).astype(np.uint32)
    assert want.max() > 1 and (want == 0).any()
    assert np.array_equal(counts.cpu().numpy().view(np.uint32), want)
    # counts only: the masks go to the scratch
    assert hz.lib.horizonator_viewshed_device(C.byref(p.h.context), len(views), p.h._eyes(views), 1.7, None,
                                              counts.data_ptr(), None)
    torch.cuda.synchronize()
    assert np.array_equal(counts.cpu().numpy().view(np.uint32), 2 * want)
    # then one view, counts only: the scratch again, at a smaller size
    one = views[5:6]
    assert hz.lib.horizonator_viewshed_device(C.byref(p.h.context), 1, p.h._eyes(one), 1.7, None,
                                              counts.data_ptr(), None)
    torch.cuda.synchronize()
    assert np.array_equal(counts.cpu().numpy().view(np.uint32), 2 * want + m[5])

    # host memory: += on the caller's counts, twice
    pattern = np.random.default_rng(5).integers(1, 1 << 20, (N, N)).astype(np.uint32)
    hc = pattern.copy()
    for rep in (1, 2):
        assert hz.lib.horizonator_viewshed(C.byref(p.h.context), len(views), p.h._eyes(views), 1.7, None,
                                           hc.ctypes.data)
        assert np.array_equal(hc, pattern + rep * want), rep
    # masks only, into host memory
    hm = np.full((len(views), N, p.w32), POISON, np.uint32)
    assert hz.lib.horizonator_viewshed(C.byref(p.h.context), len(views), p.h._eyes(views), 1.7, hm.ctypes.data, None)
    assert np.array_equal(hm, got)
    # one view after the batch: masks and counts in host memory
    hm1, hc1 = np.full((1, N, p.w32), POISON, np.uint32), pattern.copy()
    assert hz.lib.horizonator_viewshed(C.byref(p.h.context), 1, p.h._eyes(one), 1.7, hm1.ctypes.data, hc1.ctypes.data)
    assert np.array_equal(hm1[0], got[5]) and np.array_equal(hc1, pattern + m[5])


def test_the_first_counts_call_of_a_context_adds_to_the_callers_counts(hz, tiles_c1):
    """On a fresh context the host call's device counts are allocated by this call: what it adds to is still the
    caller's pattern"""
    p = Pair(hz, tiles_c1, 300, False, C1_LAT, C1_LON)
    try:
        views = _mixed_views(p)[:70]
        pattern = np.random.default_rng(9).integers(1, 1 << 20, (p.N, p.N)).astype(np.uint32)
        hc = pattern.copy()
        assert hz.lib.horizonator_viewshed(C.byref(p.h.context), len(views), p.h._eyes(views), 1.7, None,
                                           hc.ctypes.data)
        want = sum(unpack_mask(p.oracle_words(v, 1.7)[0]).astype(np.uint32) for v in views)
        assert np.array_equal(hc, pattern + want)
    finally:
        p.h.close()
        p.o.close()


def test_on_a_side_stream(pairs, tiles_c1):
    torch = _torch()
    p = pairs(tiles_c1, 300)
    views = _mixed_views(p)[:70]
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        check(p, views, 1.7, what="side stream", stream=s.cuda_stream)


# ---------------------------------------------------------------------------------------------- interleaving

def test_after_renders_and_curvature_toggles(pairs, tiles_c1):
    """Viewsheds right after a batch render on the same context, and after curvature goes off and on again, are the
    oracle's for the mode then current"""
    torch = _torch()
    p = pairs(tiles_c1, 1200)
    views = [(C1_LAT, C1_LON), p.on_vertex(1220, 1170), p.view(("below", p.N - 1), 0.3)]
    W, H = 64, 16
    rviews = [(C1_LAT + 0.01 * k, C1_LON - 0.02 * k, -180., 180.) for k in range(3)]
    img = torch.zeros((len(rviews), H, W, 3), dtype=torch.uint8, device="cuda")
    rng = torch.zeros((len(rviews), H, W), dtype=torch.float32, device="cuda")
    c = vertex.curvature(True, 0.13)
    torch.cuda.synchronize()
    try:
        p.h.render_batch_device(rviews, img.data_ptr(), rng.data_ptr())
        check(p, views, 1.7, what="after a render")
        assert (rng > 0).any().item()
        p.h.set_earth_curvature(True, 0.13)
        check(p, views, 1.7, curvature=c, what="curvature on")
        p.h.render_batch_device(rviews, img.data_ptr(), rng.data_ptr())
        check(p, views, 1.7, curvature=c, what="curvature on, after a render")
        p.h.set_earth_curvature(False)
        check(p, views, 1.7, what="curvature off again")
        p.h.set_earth_curvature(True, 0.13)
        check(p, views, 1.7, curvature=c, what="curvature on again")
    finally:
        p.h.set_earth_curvature(False)
