"""The span grid over the visibility buffer (hz_device.h): occlusion tests answered from it alone on profiled lone renders,
and renders that stay bit-identical while the grid and the keys carry what earlier renders of other views, other
widths and other epochs left behind.  Run on the B200 box: pytest -m gpu."""
import os

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON

pytestmark = pytest.mark.gpu

C2_LAT, C2_LON = 34.0 + 1.0 / 7200.0, -117.0 + 1.0 / 7200.0
FULL = (-180.05, 179.95)

LONE_VIEWS = {
    "c2": (C2_LAT, C2_LON) + FULL,
    "c5_21_42": (33.5 + 21.5 / 64 + 1.0 / 7200.0, -117.5 + 42.5 / 64 + 1.0 / 7200.0) + FULL,
    "eye3km": (C2_LAT, C2_LON) + FULL + (3000.,),
}


@pytest.fixture(scope="module")
def c2():
    import horizonator_b200 as hz
    from tools import synth
    tiles = synth.config2_tiles(os.environ.get("HZ_BENCH_TILES", "/tmp/hz_tiles_c2"))
    h = hz.horizonator(C2_LAT, C2_LON, 3600, 600, SRTM1=True, dir_dems=tiles, render_radius_m=150000.)
    h.set_zextents(100., 150000.)
    h.profile(True)
    return h


@pytest.mark.parametrize("name", sorted(LONE_VIEWS))
def test_grid_decides_occlusion(c2, name):
    """Some occluded tiles and blocks are found from the span grid alone, never more than were found occluded."""
    c2.render_batch([LONE_VIEWS[name]])
    c = c2.render_counters()
    occluded = c["tiles_occluded"] + c["blocks_occluded"]
    print("%s: %d of %d occluded rectangles from the grid alone (%.3f), %d blocks' spans recomputed"
          % (name, c["occluded_by_grid"], occluded, c["occluded_by_grid"] / max(occluded, 1), c["span_blocks"]))
    assert 0 < c["occluded_by_grid"] <= occluded
    assert c["span_blocks"] > 0


W, H, R = 720, 240, 400
# different skylines: where one has terrain the next often has sky
C1_VIEWS = [
    (C1_LAT, C1_LON, -180.05, 179.95),
    (C1_LAT + 0.03, C1_LON - 0.02, -30.0, 30.0),
    (C1_LAT, C1_LON, -180.05, 179.95, 3000.0),
    (C1_LAT - 0.04, C1_LON + 0.05, 100.0, 160.0),
]


def _context(hz, tiles):
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles, render_radius_cells=R)
    h.set_zextents(100., 100000.)
    return h


def test_reused_buffers_render_like_fresh_ones(tiles_c1):
    """17 lone renders and 17 batch calls on one context, alternating views: the epoch of the keys wraps twice on the
    lone view's buffer and on the batch views', and every render equals the same view rendered by a fresh context."""
    import horizonator_b200 as hz
    fresh = {}
    for v in C1_VIEWS:
        f = _context(hz, tiles_c1)
        img, rng = f.render_batch([v])
        fresh[v] = (img[0].copy(), rng[0].copy())
        f.close()
    h = _context(hz, tiles_c1)
    n = len(C1_VIEWS)
    for k in range(17):
        v = C1_VIEWS[k % n]
        img, rng = h.render_batch([v])
        assert np.array_equal(img[0], fresh[v][0]) and np.array_equal(rng[0], fresh[v][1]), ("lone", k, v)
        batch = [C1_VIEWS[(k + 1 + j) % n] for j in range(3)]
        img, rng = h.render_batch(batch)
        for j, b in enumerate(batch):
            assert np.array_equal(img[j], fresh[b][0]) and np.array_equal(rng[j], fresh[b][1]), ("batch", k, j, b)
    h.close()


@pytest.mark.parametrize("x0,x1", [(36, 136), (36, 137), (0, 20)])
def test_wedge_of_odd_width(tiles_c1, x0, x1):
    """Wedges whose widths are not multiples of 8 (spans and blocks cut at the wedge's edge, the grid laid out for
    another width than the previous render's) equal those columns of the whole render, and the whole render after
    them equals the one before."""
    import horizonator_b200 as hz
    h = _context(hz, tiles_c1)
    v = C1_VIEWS[0]
    img, rng = h.render(v[2], v[3], lat=v[0], lon=v[1], znear=100., zfar=100000.)
    img, rng = img.copy(), rng.copy()
    assert (rng[:, x0:x1] > 0).any()
    wi, wr = np.zeros_like(img), np.full_like(rng, -2.0)
    h.render_wedge_host(x0, x1, wi, wr)
    assert np.array_equal(wi[:, x0:x1], img[:, x0:x1]) and np.array_equal(wr[:, x0:x1], rng[:, x0:x1])
    img2, rng2 = h.render(v[2], v[3], znear=100., zfar=100000.)
    assert np.array_equal(img2, img) and np.array_equal(rng2, rng)
    h.close()
