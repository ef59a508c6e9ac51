"""The culling kernels (k_tiles, k_blocks) on profiled lone renders of the C2 context: every tile of the bands is
looked at exactly once, and every culling decision is the one recorded before k_tiles enumerated the band's ring
and the culling loops became warp-local.  A profiled chain runs k_big in line, so the visibility buffer each culling
kernel sees is fixed: a different counter means a different decision.  Run on the B200 box: pytest -m gpu."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

C2_LAT, C2_LON = 34.0 + 1.0 / 7200.0, -117.0 + 1.0 / 7200.0
FULL = (-180.05, 179.95)
TILE_CELLS, NEAR_RINGS = 32, 2          # HZ_TILE_CELLS, NEAR_RINGS of the library


def _c5(j, i, g=64):
    return (33.5 + (j + 0.5) / g + 1.0 / 7200.0, -117.5 + (i + 0.5) / g + 1.0 / 7200.0) + FULL


VIEWS = {
    "c2": (C2_LAT, C2_LON) + FULL,
    "c5_0_0": _c5(0, 0),
    "c5_21_42": _c5(21, 42),
    "c5_42_21": _c5(42, 21),
    "c5_63_63": _c5(63, 63),
    "eye3km": (C2_LAT, C2_LON) + FULL + (3000.,),
    "zoom10": (C2_LAT, C2_LON, 40., 50.),
}
# eyes within two tiles of an edge and in corners (tile column, tile row; negative: from the far edge)
EYE_TILES = {"west_edge": (1, 183), "north_edge": (200, -2), "sw_corner": (0, 0), "ne_corner": (-1, -1)}


def c2_context():
    import horizonator_b200 as hz
    from tools import synth
    tiles = synth.config2_tiles(os.environ.get("HZ_BENCH_TILES", "/tmp/hz_tiles_c2"))
    h = hz.horizonator(C2_LAT, C2_LON, 3600, 600, SRTM1=True, dir_dems=tiles, render_radius_m=150000.)
    h.set_zextents(100., 150000.)
    h.profile(True)
    return h


def counters(h, view):
    h.render_batch([view])
    return h.render_counters()


def n_tiles(h):
    """Tiles per side of the mesh: the N - 1 cells of its N = 2R vertices per side, 32 to a tile."""
    return (2 * h._ctx.dems.radius_cells - 1 + TILE_CELLS - 1) // TILE_CELLS


def eye_tile(h, lat, lon):
    """The eye's tile as the library computes it (compute_move, then the tile of the viewer cell), in float32."""
    d = h._ctx.dems
    f = np.float32
    vci = (f(lon) - f(d.origin_dem_lon_lat[0])) * f(d.cells_per_deg) - f(d.origin_dem_cellij[0])
    vcj = (f(lat) - f(d.origin_dem_lon_lat[1])) * f(d.cells_per_deg) - f(d.origin_dem_cellij[1])
    nt = n_tiles(h)
    return (min(max(int(np.floor(vci / f(TILE_CELLS))), 0), nt - 1), min(max(int(np.floor(vcj / f(TILE_CELLS))), 0), nt - 1))


def view_at_tile(h, ti, tj):
    """A full-circle view whose eye sits in the middle of tile (ti, tj)."""
    d, nt = h._ctx.dems, n_tiles(h)
    ti, tj = ti % nt, tj % nt
    ci, cj = ti * TILE_CELLS + TILE_CELLS // 2, tj * TILE_CELLS + TILE_CELLS // 2
    lon = d.origin_dem_lon_lat[0] + (ci + 0.5 + d.origin_dem_cellij[0]) / d.cells_per_deg
    lat = d.origin_dem_lon_lat[1] + (cj + 0.5 + d.origin_dem_cellij[1]) / d.cells_per_deg
    assert eye_tile(h, lat, lon) == (ti, tj)
    return (lat, lon) + FULL


# render_counters() of the views above, recorded on a B200 with the library as it was before the culling kernels'
# loops became warp-local (ring_*: the eyes of EYE_TILES; c2_lod: c2 with set_lod(0.5)).  All but big_entries: which
# triangles k_raster hands to k_big depends on which others share their warp, i.e. on the order of the triangle list,
# which atomics decide (it differed between two runs of the same library).
CULLING = ("tiles", "tiles_far", "tiles_window", "tiles_occluded", "blocks", "blocks_far", "blocks_window",
           "blocks_occluded", "blocks_meshed", "triangles")
EXPECTED = {
    "c2": (134664, 45965, 20744, 61895, 389384, 1475, 226967, 122876, 38066, 128106),
    "c5_0_0": (134664, 58336, 16948, 52067, 469632, 6593, 270218, 147453, 45368, 121116),
    "c5_21_42": (134664, 47738, 20604, 61948, 281480, 261, 134609, 109054, 37556, 142304),
    "c5_42_21": (134664, 47603, 20305, 49864, 1082688, 6232, 768227, 68403, 239826, 438909),
    "c5_63_63": (134664, 57451, 19472, 36595, 1348896, 2761, 918296, 110927, 316912, 490064),
    "eye3km": (134664, 45965, 14974, 669, 4676792, 51282, 3563384, 4601, 1057525, 2160816),
    "zoom10": (134664, 45965, 85176, 1, 226952, 2235, 64797, 3793, 156127, 1852083),
    "ring_west_edge": (134669, 89838, 9747, 7088, 1793024, 23466, 1330226, 35470, 403862, 612959),
    "ring_north_edge": (134669, 90020, 10688, 25567, 534800, 2381, 350921, 25535, 155963, 406657),
    "ring_sw_corner": (134680, 112729, 3968, 16229, 112832, 123, 46427, 46157, 20125, 72585),
    "ring_ne_corner": (134680, 111862, 5669, 13904, 198337, 703, 125414, 28414, 43806, 90033),
    "c2_lod": (134664, 45751, 20868, 63001, 268698, 10, 125739, 115360, 27589, 122579),
}


@pytest.fixture(scope="module")
def c2():
    return c2_context()


@pytest.mark.parametrize("where", sorted(EYE_TILES))
def test_every_tile_of_the_bands_is_looked_at_once(c2, where):
    """The bands cover the mesh outside the near tiles: `tiles` is the mesh's tile count minus the near square
    around the eye's tile, clipped to the mesh."""
    nt = n_tiles(c2)
    view = view_at_tile(c2, *EYE_TILES[where])
    ti, tj = eye_tile(c2, view[0], view[1])
    near_w = min(ti + NEAR_RINGS, nt - 1) - max(ti - NEAR_RINGS, 0) + 1
    near_h = min(tj + NEAR_RINGS, nt - 1) - max(tj - NEAR_RINGS, 0) + 1
    assert counters(c2, view)["tiles"] == nt * nt - near_w * near_h


def test_centre_ring_coverage(c2):
    assert n_tiles(c2) == 367
    assert counters(c2, VIEWS["c2"])["tiles"] == 367 * 367 - 5 * 5


@pytest.mark.parametrize("name", sorted(VIEWS) + ["ring_" + k for k in sorted(EYE_TILES)] + ["c2_lod"])
def test_culling_decisions_unchanged(c2, name):
    if name == "c2_lod":
        c2.set_lod(0.5)
        try:
            got = counters(c2, VIEWS["c2"])
        finally:
            c2.set_lod(0.)
    elif name.startswith("ring_"):
        got = counters(c2, view_at_tile(c2, *EYE_TILES[name[5:]]))
    else:
        got = counters(c2, VIEWS[name])
    assert tuple(got[k] for k in CULLING) == EXPECTED[name]
