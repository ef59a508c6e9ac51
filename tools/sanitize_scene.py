"""One mid-size scene through every kernel and host path, for compute-sanitizer: single renders (wide and zoomed-in:
near pass, bands, large triangles, middle-sized triangles), a batch of 11 views in chunks of 8 and 3 with a view
dimension on two view sets, pageable and page-locked destinations, a wedge into a host panorama, the horizon profile."""
import os, sys, tempfile
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import horizonator_b200 as hz
from tools import synth
d = synth.config1_tiles(os.path.join(tempfile.gettempdir(), "hz_smoke_tiles"))
lat, lon = 35.0 + 1.0 / 2400.0, -117.0 + 1.0 / 2400.0
W, H = 720, 120
h = hz.horizonator(lat, lon, W, H, dir_dems=d, render_radius_cells=400)
a = h.render(-180.05, 179.95, zfar=100000.)
z = h.render(40., 46., zfar=100000.)
assert (z[1] > 0).mean() > 0.5
h.set_zextents(100., 100000.)
views = [(lat, lon, -180.05, 179.95), (lat + 0.01, lon, -90., 90.), (lat, lon + 0.01, 0., 45.), (lat, lon, 40., 46.)]
views += [(lat + 0.002 * k, lon - 0.003 * k, -180.05, 179.95, 1500. + 100 * k) for k in range(7)]
bi, br = h.render_batch(views)
assert np.array_equal(bi[0], a[0]) and np.array_equal(br[0], a[1])
assert np.array_equal(bi[3], z[0]) and np.array_equal(br[3], z[1])
pi, pr = np.zeros((H, W, 3), np.uint8), np.zeros((H, W), np.float32)       # pageable: the staged copy pipeline
h.pan_zoom(-180.05, 179.95); h.move(lat, lon)
h.render_into(pi, pr)
assert np.array_equal(pi, a[0]) and np.array_equal(pr, a[1])
wi, wr = np.zeros((H, W, 3), np.uint8), np.zeros((H, W), np.float32)
for x0, x1 in ((0, 240), (240, 481), (481, W)):
    h.render_wedge_host(x0, x1, wi, wr)
assert np.array_equal(wi, a[0]) and np.array_equal(wr, a[1])
print("ok", h.last_render_stats())
