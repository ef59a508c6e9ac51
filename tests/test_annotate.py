"""Labels of points of interest (horizonator_annotate_batch*, include/horizonator-batch.h), checked without a GPU: the
ctypes mirrors of horizonator_poi_t / horizonator_label_t against a compiled probe of the header, and the host
restatement of the rule (oracle/annotate.py, which the GPU tests compare the kernel with) on known answers."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import annotate as oa

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GCC = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"

PROBE = r"""
#include <stddef.h>
#include <stdio.h>
#include "horizonator-batch.h"
int main(void)
{
    printf("poi %zu %zu %zu %zu\n", sizeof(horizonator_poi_t), offsetof(horizonator_poi_t, lat),
           offsetof(horizonator_poi_t, lon), offsetof(horizonator_poi_t, ele));
    printf("label %zu %zu %zu %zu %zu\n", sizeof(horizonator_label_t), offsetof(horizonator_label_t, x),
           offsetof(horizonator_label_t, y), offsetof(horizonator_label_t, range_m),
           offsetof(horizonator_label_t, range_rendered_m));
    return 0;
}
"""


def test_ctypes_mirrors_match_the_header(tmp_path):
    import horizonator_b200 as hz
    src, exe = tmp_path / "probe.c", tmp_path / "probe"
    src.write_text(PROBE)
    subprocess.run([GCC, "-std=gnu99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = {line.split()[0]: [int(v) for v in line.split()[1:]]
           for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()}
    assert got["poi"] == [24, 0, 8, 16]
    assert got["label"] == [16, 0, 4, 8, 12]
    assert C.sizeof(hz.poi_t) == 24 and [hz.poi_t.lat.offset, hz.poi_t.lon.offset, hz.poi_t.ele.offset] == [0, 8, 16]
    assert C.sizeof(hz.label_t) == 16
    assert [getattr(hz.label_t, f).offset for f in ("x", "y", "range_m", "range_rendered_m")] == [0, 4, 8, 12]
    assert hz.LABEL_DTYPE.itemsize == 16 and list(hz.LABEL_DTYPE.names) == list(oa.LABEL_DTYPE.names)
    assert [hz.LABEL_DTYPE.fields[f][1] for f in hz.LABEL_DTYPE.names] == [0, 4, 8, 12]


# ---- the vertical search on synthetic range images

H, W = 40, 30


def _image(col=10, rows=None):
    """Sky everywhere; in column `col`, rows -> range."""
    r = np.full((H, W), -1.0, np.float32)
    for row, v in (rows or {}).items():
        r[row, col] = v
    return r


def test_poi_exactly_on_a_rendered_range_is_visible():
    img = _image(rows={20: 5000.0, 21: 4900.0, 22: 4800.0})
    vis, best, have = oa.search(img, 10.2, 20.3, 5000.0)
    assert vis and best == 0 and have == np.float32(5000.0)
    # a search that starts above the match walks down to it: the error shrinks until row 21, then grows
    vis, best, have = oa.search(img, 10.0, 17.0, 4900.0)
    assert vis and best == 4 and have == np.float32(4900.0)


@pytest.mark.parametrize("err,visible", [(499.0, True), (501.0, False), (500.0, False)])
def test_range_fuzz_is_500_m(err, visible):
    img = _image(rows={20: 10000.0})
    vis, best, have = oa.search(img, 10.0, 20.0, 10000.0 + err)
    assert vis == visible
    assert (have == np.float32(10000.0)) if visible else have is None


@pytest.mark.parametrize("rng,gated", [(499.99, True), (500.0, False), (100000.0, False), (100000.01, True)])
def test_distance_gates(rng, gated):
    img = _image(rows={20: np.float32(rng)})
    vis, _, _ = oa.search(img, 10.0, 20.0, rng)
    assert (vis is None) == gated
    if not gated:
        assert vis


@pytest.mark.parametrize("x,inside", [(-0.5, False), (-0.49, True), (29.49, True), (29.5, False)])
def test_column_gate_is_lround_x_in_the_image(x, inside):
    col = min(max(int(math.floor(x + 0.5)), 0), W - 1)
    img = _image(col=col, rows={20: 3000.0})
    vis, _, _ = oa.search(img, x, 20.0, 3000.0)
    assert (vis is not None) == inside


def test_lround_is_half_away_from_zero():
    assert [oa._lround(v) for v in (-0.5, -0.49, 0.49999999999999994, 0.5, 1.5, 2.5, -1.5)] == [-1, 0, 0, 1, 2, 3, -2]


def test_first_rows_clip_the_search_at_the_top():
    # y = 2.3: d = -6 .. -3 give y + d < 0 and are skipped; row 0 is reached at d = -2
    img = _image(rows={0: 7000.0, 1: 6000.0})
    vis, best, have = oa.search(img, 10.0, 2.3, 7100.0)
    assert vis and best == -2 and have == np.float32(7000.0)
    # y + d = -0.2 < 0 skips d = -3 even though lround(y) + d = 0 would be a row
    img = _image(rows={0: 7000.0})
    vis, _, _ = oa.search(img, 10.0, 2.8, 7000.0)
    assert vis is False


def test_last_rows_stop_the_search_at_the_bottom():
    img = _image(rows={H - 1: 900.0})
    vis, best, have = oa.search(img, 10.0, H - 3.0, 900.0)
    assert vis and best == 2
    vis, best, _ = oa.search(img, 10.0, H - 1.4, 900.0)
    assert vis and best == 0
    # y = H - 0.4: lround(y) = H, so d = 0 is below the image (skipped) and d = 1 ends the search (y + 1 >= H)
    vis, best, _ = oa.search(img, 10.0, H - 0.4, 900.0)
    assert vis and best == -1 and oa._lround(H - 0.4) == H


def test_search_stops_as_soon_as_the_error_grows():
    # rows 14.. : 8000 (err 3000), 6000 (err 1000), 9000 (err 4000: stop), 5000 (exact, never reached)
    img = _image(rows={14: 8000.0, 15: 6000.0, 16: 9000.0, 17: 5000.0})
    vis, best, _ = oa.search(img, 10.0, 20.0, 5000.0)
    assert vis is False and best == -5
    # an equal error also stops it (only a smaller one moves on)
    img = _image(rows={14: 5400.0, 15: 4600.0, 16: 5000.0})
    vis, best, have = oa.search(img, 10.0, 20.0, 5000.0)
    assert vis and best == -6 and have == np.float32(5400.0)


def test_sky_rows_are_skipped_not_stopped_at():
    img = _image(rows={14: 8000.0, 18: 5000.0})
    vis, best, have = oa.search(img, 10.0, 20.0, 5000.0)
    assert vis and best == -2 and have == np.float32(5000.0)


# ---- the whole rule with the product's projection

@pytest.fixture(scope="module")
def project():
    import horizonator_b200 as hz
    return hz.lib.horizonator_project


def _latlon_at(lat0, lon0, az_deg, dist):
    cos_lat = math.cos(float(np.float32(lat0)) * math.pi / 180.)
    north, east = dist * math.cos(math.radians(az_deg)), dist * math.sin(math.radians(az_deg))
    return (float(np.float32(lat0)) + north / 6371000.0 * 180. / math.pi,
            float(np.float32(lon0)) + east / 6371000.0 / cos_lat * 180. / math.pi)


def test_outside_the_window_gives_minus_one_everywhere(project):
    lat0, lon0, eye = 35.0, -117.0, 1000.0
    img = np.full((H, W), 4000.0, np.float32)
    behind = _latlon_at(lat0, lon0, 180.0, 4000.0)             # azimuth outside -45 .. 45
    above = _latlon_at(lat0, lon0, 0.0, 4000.0)                # elevation far above the window
    pois = [(behind[0], behind[1], eye), (above[0], above[1], eye + 20000.0)]
    out = oa.annotate_view(project, img, pois, lat0, lon0, eye, -45.0, 45.0)
    assert (out.labels.view(np.float32) == -1.0).all() and not out.visible.any()


def test_a_poi_on_the_terrain_as_rendered_is_labelled(project):
    lat0, lon0, eye = 35.0, -117.0, 1000.0
    la, lo = _latlon_at(lat0, lon0, 10.0, 5000.0)
    pois = [(la, lo, eye + 30.0)]
    probe = oa.annotate_view(project, np.full((H, W), -1.0, np.float32), pois, lat0, lon0, eye, -45.0, 45.0)
    x, y, rng = probe.x[0], probe.y[0], probe.range[0]
    assert 0 <= x < W and 0 <= y < H and probe.labels["range_rendered_m"][0] == -1.0
    img = np.full((H, W), -1.0, np.float32)
    img[oa._lround(y) + 1, oa._lround(x)] = np.float32(rng + 100.0)
    out = oa.annotate_view(project, img, pois, lat0, lon0, eye, -45.0, 45.0)
    lab = out.labels[0]
    assert out.visible[0] and out.best[0] == 1
    assert lab["x"] == np.float32(x) and lab["range_m"] == np.float32(rng)
    assert lab["y"] == np.float32(y + 1.0) and lab["range_rendered_m"] == np.float32(rng + 100.0)
