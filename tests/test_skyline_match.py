"""Skylines and their match against an observed skyline (horizonator_skyline_match*, include/horizonator-batch.h),
checked without a GPU: the ctypes mirror of horizonator_skyline_sample_t against a compiled probe of the header, the
host restatement of the scoring rule (oracle/skyline_match.py, which the GPU tests compare the kernel with) on
hand-made skylines, and the samples' formula against the library's host horizonator_project()."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import skyline_match as om

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GCC = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"

PROBE = r"""
#include <stddef.h>
#include <stdio.h>
#include "horizonator-batch.h"
int main(void)
{
    printf("%zu %zu %zu\n", sizeof(horizonator_skyline_sample_t), offsetof(horizonator_skyline_sample_t, dx),
           offsetof(horizonator_skyline_sample_t, y));
    return 0;
}
"""


def test_ctypes_mirror_matches_the_header(tmp_path):
    import horizonator_b200 as hz
    src, exe = tmp_path / "probe.c", tmp_path / "probe"
    src.write_text(PROBE)
    subprocess.run([GCC, "-std=gnu99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [8, 0, 4]
    assert C.sizeof(hz.skyline_sample_t) == 8
    assert [hz.skyline_sample_t.dx.offset, hz.skyline_sample_t.y.offset] == [0, 4]
    assert hz.SKYLINE_SAMPLE_DTYPE == om.SAMPLE_DTYPE and hz.SKYLINE_SAMPLE_DTYPE.itemsize == 8


# ---- the rule on hand-made skylines

W = 12


def test_flat_skyline_matches_at_every_heading():
    rows = np.full((1, W), 5, np.int64)
    got = om.scores(rows, om.samples([(d, 4.5) for d in range(-3, 4)]), 8.0, True)
    assert (got == 0.0).all()
    # 1.25 rows off everywhere
    got = om.scores(rows, om.samples([(0, 3.25), (2, 5.75)]), 8.0, True)
    assert (got == np.float32(1.25)).all()


def test_a_step_is_found_at_its_shift():
    rows = np.where(np.arange(W) < 6, 10, 3)[None, :]
    # the observed step: columns dx = 0..3 at row 10, dx = 4..7 at row 3 (edges half a row above)
    smp = om.samples([(d, 9.5 if d < 4 else 2.5) for d in range(8)])
    got = om.scores(rows, smp, 8.0, False)[0]
    assert got[2] == 0.0 and np.argmin(got) == 2 and (got[np.arange(W) != 2] > 0).all()


def test_wrap_against_no_wrap_at_both_ends():
    rows = np.arange(W)[None, :] % 4
    smp = om.samples([(-1, rows[0, W - 1] - 0.5), (1, rows[0, 1] - 0.5)])
    wrap = om.scores(rows, smp, 8.0, True)[0]
    flat = om.scores(rows, smp, 8.0, False)[0]
    # h = 0: c = -1 wraps to W-1 (exact) / is missing; c = 1 exact on both
    assert wrap[0] == 0.0 and flat[0] == np.float32(4.0)
    # h = W-1: c = W wraps to 0 (rows 0, y = rows[1] - 0.5 = 0.5: error 1) / is missing
    assert wrap[W - 1] == np.float32((abs((rows[0, W - 2] - 0.5) - (rows[0, W - 1] - 0.5)) + 1.0) / 2)
    assert flat[W - 1] == np.float32((abs((rows[0, W - 2] - 0.5) - (rows[0, W - 1] - 0.5)) + 8.0) / 2)


def test_all_sky_columns_cost_clip_rows():
    rows = np.full((2, W), 7, np.int64)
    rows[1, 3] = -1
    smp = om.samples([(0, 6.5)])
    got = om.scores(rows, smp, 3.0, True)
    assert (got[0] == 0.0).all()
    assert got[1, 3] == np.float32(3.0) and (np.delete(got[1], 3) == 0.0).all()


@pytest.mark.parametrize("y,want", [(6.5 - 2.0, 2.0), (6.5 + 2.5, 2.5), (6.5 - 2.75, 2.75), (6.5 + 3.0, 2.75),
                                    (6.5 - 100.0, 2.75)])
def test_errors_above_and_below_clip_rows(y, want):
    rows = np.full((1, W), 7, np.int64)
    got = om.scores(rows, om.samples([(0, y)]), 2.75, True)
    assert (got == np.float32(want)).all()


@pytest.mark.parametrize("dx", [-W, -W - 5, -3 * W + 2, W, W + 3, 5 * W - 1, -(2 ** 31), 2 ** 31 - 1])
def test_negative_and_beyond_width_offsets(dx):
    rows = (np.arange(W) * 3 % 11)[None, :]
    smp = om.samples([(dx, 4.0)])
    wrap = om.scores(rows, smp, 8.0, True)[0]
    flat = om.scores(rows, smp, 8.0, False)[0]
    c = (np.arange(W) + dx) % W
    assert np.array_equal(wrap, np.fmin(np.abs((rows[0, c] - np.float32(0.5)) - np.float32(4.0)), 8.0).astype(np.float32))
    assert (flat == np.float32(8.0)).all()           # |dx| >= W: every column is missing


def test_the_sum_runs_in_sample_order_in_float32():
    rows = np.zeros((1, 1), np.int64)
    # errors 2^24 - 1 (clip), then 1, 1, 1: added in order in float32 each 1 is lost or kept exactly as fp32 does
    big = np.float32(2 ** 24)
    smp = om.samples([(0, -0.5 - float(big))] + [(0, -1.5)] * 3)
    got = om.scores(rows, smp, float(big), True)[0, 0]
    acc = np.float32(0)
    for d in (big, np.float32(1), np.float32(1), np.float32(1)):
        acc = np.float32(acc + d)
    assert got == np.float32(acc / np.float32(4))


# ---- the samples' formula against horizonator_project()

def _latlon_at(lat0, lon0, az_deg, dist):
    """the point `dist` metres from the eye at azimuth az_deg, by the inverse of horizonator_project()'s flat-earth east /
    north"""
    cos_lat = math.cos(lat0 * math.pi / 180.)
    north, east = dist * math.cos(math.radians(az_deg)), dist * math.sin(math.radians(az_deg))
    return lat0 + north / (6371000.0 * math.pi / 180), lon0 + east / (6371000.0 * cos_lat * math.pi / 180)


@pytest.mark.parametrize("Wp,Hp,az0,width", [(3600, 600, -180.0, 359.9), (1200, 300, 30.0, 60.0), (640, 480, -20.0, 5.0)])
def test_samples_agree_with_horizonator_project(Wp, Hp, az0, width):
    import horizonator_b200 as hz
    lat0, lon0, ele0 = 35.2, -117.3, 1500.0
    p = width / Wp
    rs = np.random.default_rng(Wp)
    h = int(Wp // 3)
    heading = az0 + (h + 0.5) * p                       # the heading of column h
    # angles within the window, column offsets away from half-integers (rint's ties)
    rel = (rs.integers(-h + 2, Wp - h - 2, 40) + rs.uniform(-0.4, 0.4, 40)) * p
    el = rs.uniform(-0.45, 0.45, 40) * Hp * p
    smp = hz.skyline_samples(rel, el, width, Wp, Hp)
    x, y, r = C.c_double(), C.c_double(), C.c_double()
    for k in range(len(rel)):
        dist = 8000.0 + 500.0 * k
        la, lo = _latlon_at(lat0, lon0, heading + rel[k], dist)
        ele = ele0 + dist * math.tan(math.radians(el[k]))
        assert hz.lib.horizonator_project(C.byref(x), C.byref(y), C.byref(r), lat0, math.cos(lat0 * math.pi / 180.),
                                          lon0, ele0, la, lo, ele, az0 * math.pi / 180., (az0 + width) * math.pi / 180.,
                                          Wp, Hp)
        want_y = (Hp - 1) / 2. - el[k] / p
        assert abs(y.value - want_y) < 1e-9, (k, y.value, want_y)
        assert smp["y"][k] == np.float32(want_y)
        assert int(np.rint(x.value)) - h == smp["dx"][k], (k, x.value, smp["dx"][k])
