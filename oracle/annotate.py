"""oracle/annotate.py -- TEST INFRASTRUCTURE.  A host restatement of the labels rule of include/horizonator-batch.h
(horizonator_annotate_batch*), which is the command-line tool's write_labels() (cli/horizonator-standalone.c) and the
reference's annotator.c:280-348, applied to a range image.

Only tests/ and tools/ may import this.  The projection is the product's own horizonator_project() through ctypes: that
function is pinned bit for bit against the reference's elsewhere (tests/test_host_logic.py), and what is restated here is
everything around it -- the inputs as the library forms them, the gates and the vertical search.

    search(ranges, x, y, rng)                     -> (visible, best, rendered range)  for one projected POI
    annotate_view(project, ranges, pois, lat, lon, eye_z, az_deg0, az_deg1)   -> Labels of one view
"""
import ctypes as C
import math

import numpy as np

MARKER_DIST_MIN = 500.0          # annotator.c:19-23
MARKER_DIST_MAX = 100000.0
MARKER_RANGE_FUZZ = 500.0
MARKER_PIXEL_FUZZ = 6

LABEL_DTYPE = np.dtype([("x", np.float32), ("y", np.float32), ("range_m", np.float32), ("range_rendered_m", np.float32)])


def _lround(v):
    """C lround(): half away from zero (v - floor(v) is exact, v + 0.5 is not)."""
    if v < 0:
        return -_lround(-v)
    f = math.floor(v)
    return int(f) + (1 if v - f >= 0.5 else 0)


def search(ranges, x, y, rng):
    """The gates and the vertical search of write_labels() for a POI projected to (x, y) at range `rng` (doubles) over
    a range image (H, W) float32, top row first, <= 0 where no terrain.  Returns (visible, best offset, the rendered
    range matched (float32) or None); visible is None where a gate drops the POI before the search."""
    H, W = ranges.shape
    if rng < MARKER_DIST_MIN or rng > MARKER_DIST_MAX:
        return None, 0, None
    col = _lround(x)
    if col < 0 or col >= W:
        return None, 0, None
    best, best_err, have_best = 0, float(np.finfo(np.float64).max), None
    for d in range(-MARKER_PIXEL_FUZZ, MARKER_PIXEL_FUZZ):
        if y + float(d) < 0:
            continue
        if y + float(d) >= H:
            break
        r = _lround(y) + d
        if r < 0 or r >= H:
            continue
        have = ranges[r, col]
        if have <= np.float32(0.0):
            continue
        err = abs(rng - float(have))
        if err < best_err:
            best_err, best, have_best = err, d, have
        else:
            break                                   # ranges only get nearer further down
    if best_err >= MARKER_RANGE_FUZZ:
        return False, best, None
    return True, best, have_best


class Labels:
    """One view's labels: `labels` (m,) LABEL_DTYPE as the library returns them, and the double-precision values they
    were rounded from (x, y, range; NaN outside the window), the visibility and the search offset per POI."""

    def __init__(self, m):
        self.labels = np.full(m, -1.0, np.float32).repeat(4).view(LABEL_DTYPE)
        self.x = np.full(m, np.nan)
        self.y = np.full(m, np.nan)
        self.range = np.full(m, np.nan)
        self.visible = np.zeros(m, bool)
        self.best = np.zeros(m, int)


def view_inputs(lat, lon, eye_z, az_deg0, az_deg1):
    """The projection's inputs of a view as the library forms them from horizonator_view_t (floats) and the eye height."""
    lat_d, lon_d = float(np.float32(lat)), float(np.float32(lon))
    return (lat_d, math.cos(lat_d * math.pi / 180.), lon_d, float(np.float32(eye_z)),
            float(np.float32(az_deg0)) * math.pi / 180., float(np.float32(az_deg1)) * math.pi / 180.)


def annotate_view(project, ranges, pois, lat, lon, eye_z, az_deg0, az_deg1):
    """Labels of (m, 3) POIs (lat, lon, ele) for one view whose range image is `ranges` (H, W).  project: the
    product's horizonator_project (ctypes function with its argtypes declared)."""
    H, W = ranges.shape
    lat_d, cos_lat, lon_d, ele, az0, az1 = view_inputs(lat, lon, eye_z, az_deg0, az_deg1)
    pois = np.asarray(pois, np.float64).reshape(-1, 3)
    out = Labels(len(pois))
    x, y, rng = C.c_double(), C.c_double(), C.c_double()
    for i, (plat, plon, pele) in enumerate(pois):
        if not project(C.byref(x), C.byref(y), C.byref(rng), lat_d, cos_lat, lon_d, ele, float(plat), float(plon),
                       float(pele), az0, az1, W, H):
            continue
        out.x[i], out.y[i], out.range[i] = x.value, y.value, rng.value
        lab = out.labels
        lab["x"][i], lab["y"][i], lab["range_m"][i] = np.float32(x.value), np.float32(y.value), np.float32(rng.value)
        visible, best, have = search(ranges, x.value, y.value, rng.value)
        if visible:
            out.visible[i], out.best[i] = True, best
            lab["y"][i] = np.float32(y.value + float(best))
            lab["range_rendered_m"][i] = have
    return out
