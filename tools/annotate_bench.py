#!/usr/bin/env python
"""annotate_bench.py -- views/s of the labels calls (horizonator_annotate_batch*) on one B200, one JSON line.

    python tools/annotate_bench.py [--out profiles/<name>.json] [--min-seconds S]

Workload: the C2 DEM and image of bench.py (synthetic SRTM1 4x4 tiles, 150 km radius, 3600 x 600; the bench's window
less a tenth of a degree, -180.05 .. 179.85, since over exactly 360 degrees horizonator_project() places no POI), 256
views per call, two view sets: `bench` (the bench viewpoint, 256 times) and `c5` (256 distinct viewpoints of bench.py's
C5 grid, every 16th); POI sets of 1 000 and 10 000 summits (vertices that are the highest of their 9 x 9 neighbourhood,
drawn with a fixed seed from the whole square).  Per combination:
  a_host_labels     horizonator_annotate_batch: POIs and labels in host memory, no panorama
  b_device_labels   horizonator_annotate_batch_device, labels only (no image, no range image)
  c_ranges_to_host  the same answer the old way: horizonator_render_batch ranges into page-locked host memory, then the
                    labels on the host (write_labels()'s rule vectorised with numpy over all POIs of a view)
  d_device_ranges   horizonator_render_batch_device, range images into HBM: the render alone, the ceiling
Each is timed with CUDA events around whole calls (c: around the render call and the host labels) on one stream after
one warm-up call, repeated until at least --min-seconds have passed.  The card's name, power limit and clocks are read
in the same run.  c's labels are compared with a's (the share of equal visibility decisions is reported).
"""
import argparse
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402  (C2, c5_grid, the tile directory)
from tools.viewshed_bench import timed  # noqa: E402


def _lround(v):
    return np.where(v < 0, -np.floor(-v + 0.5), np.floor(v + 0.5)).astype(np.int64)


def host_labels(ranges, pois, lat, lon, eye, az_deg0, az_deg1):
    """write_labels()'s rule (include/horizonator-batch.h) for one view, vectorised: (m, 4) float32 labels.  The
    projection is horizonator_project()'s formulas in numpy double (numpy's arctan2, not necessarily glibc's ulp)."""
    H, W = ranges.shape
    lat_v, lon_v = float(np.float32(lat)), float(np.float32(lon))
    cos_lat = math.cos(lat_v * math.pi / 180.)
    az0, az1 = float(np.float32(az_deg0)) * math.pi / 180., float(np.float32(az_deg1)) * math.pi / 180.
    rearth = float(np.float32(6371000.0))
    east = (pois[:, 1] - lon_v) * math.pi / 180 * rearth * cos_lat
    north = (pois[:, 0] - lat_v) * math.pi / 180 * rearth
    d2 = east * east + north * north

    def unwrap(x, near):
        d = (x - near) / (2. * math.pi)
        a = np.abs(d)
        f = np.floor(a)
        rd = np.copysign(f + (a - f >= 0.5), d)          # C round(): half away from zero
        return (d - rd) * 2. * math.pi + near
    az1u = float(unwrap(np.float64(az1 - az0), math.pi)) + az0
    center = (az0 + az1u) / 2.
    if az1u == az0:                          # a window of exactly 360 degrees: horizonator_project() places nothing
        return np.full((len(pois), 4), -1.0, np.float32)
    per_rad = 2.0 / (az1u - az0)
    az_ndc = (unwrap(np.arctan2(east, north), center) - center) * per_rad
    h = pois[:, 2] - float(np.float32(eye))
    rng = np.sqrt(d2 + h * h)
    el_ndc = np.arctan2(h, np.sqrt(d2)) * (W / H) * per_rad
    ok = (-1 <= az_ndc) & (az_ndc <= 1) & (-1 <= el_ndc) & (el_ndc <= 1)
    x = (az_ndc + 1.) / 2. * W - 0.5
    y = (-el_ndc + 1.) / 2. * H - 0.5
    out = np.full((len(pois), 4), -1.0, np.float32)
    out[ok, 0], out[ok, 1], out[ok, 2] = x[ok], y[ok], rng[ok]
    col = _lround(x)
    live = ok & (rng >= 500.) & (rng <= 100000.) & (col >= 0) & (col < W)
    best = np.zeros(len(pois), np.int64)
    best_err = np.full(len(pois), np.inf)
    have_best = np.full(len(pois), -1.0, np.float32)
    searching = live.copy()
    ry = _lround(y)
    for d in range(-6, 6):
        above = y + d < 0
        stop = (y + d >= H) & ~above
        searching &= ~stop
        r = ry + d
        step = searching & ~above & (r >= 0) & (r < H)
        have = np.where(step, ranges[np.clip(r, 0, H - 1), np.clip(col, 0, W - 1)], np.float32(-1.0))
        step &= have > 0
        err = np.abs(rng - have.astype(np.float64))
        better = step & (err < best_err)
        best_err = np.where(better, err, best_err)
        best = np.where(better, d, best)
        have_best = np.where(better, have, have_best)
        searching &= ~(step & ~better)
    vis = live & (best_err < 500.)
    out[vis, 1] = (y + best)[vis]
    out[vis, 3] = have_best[vis]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--min-seconds", type=float, default=2.0)
    args = ap.parse_args()

    import torch
    import horizonator_b200 as hz
    from tools import synth
    from tools.pois import summits
    assert torch.cuda.is_available(), "annotate_bench measures on the GPU only"
    C2 = bench.C2
    tiles = synth.config2_tiles(bench.TILES_DIR)
    W, H = C2["W"], C2["H"]
    h = hz.horizonator(C2["lat"], C2["lon"], W, H, SRTM1=True, dir_dems=tiles, render_radius_m=C2["radius_m"])
    h.set_zextents(C2["znear"], C2["zfar"])
    n = 256
    view_sets = {
        "bench": [(C2["lat"], C2["lon"], C2["az0"], C2["az1"] - 0.1)] * n,
        "c5": [(la, lo, C2["az0"], C2["az1"] - 0.1) for la, lo in bench.c5_grid(1, 0)[::16]][:n],
    }
    mosaic = h.mosaic()
    poi_sets = {m: summits(h, m, seed=m, mosaic=mosaic) for m in (1000, 10000)}
    del mosaic
    stream = torch.cuda.Stream()
    s = stream.cuda_stream
    d_ranges = torch.empty((n, H, W), dtype=torch.float32, device="cuda")
    h_ranges = hz.pinned_array((n, H, W), np.float32)
    results = {}
    with torch.cuda.stream(stream):
        for vname, views in view_sets.items():
            eyes = [h.move(v[0], v[1]) for v in views]
            for m, pois in poi_sets.items():
                d_pois = torch.as_tensor(pois, device="cuda")
                d_labels = torch.empty((n, m, 4), dtype=torch.float32, device="cuda")
                host = {}

                def a():
                    host["a"] = h.annotate(views, pois)

                def b():
                    h.annotate_device(views, d_pois, d_labels, stream=s)

                def c():
                    if not hz.lib.horizonator_render_batch(C_ctx(h), n, h._views(views), None, h_ranges.ctypes.data):
                        raise RuntimeError("horizonator_render_batch() failed")
                    host["c"] = np.stack([host_labels(h_ranges[k], pois, v[0], v[1], eyes[k], v[2], v[3])
                                          for k, v in enumerate(views)])

                def d():
                    h.render_batch_device(views, 0, d_ranges.data_ptr(), s)

                row = {}
                for name, fn in (("a_host_labels", a), ("b_device_labels", b), ("c_ranges_to_host", c),
                                 ("d_device_ranges", d)):
                    ms, reps = timed(fn, stream, args.min_seconds)
                    row[name] = {"ms_per_call": ms, "calls_timed": reps, "views_per_s": n / ms * 1e3}
                    print(vname, m, name, json.dumps(row[name]), file=sys.stderr, flush=True)
                torch.cuda.synchronize()
                la = host["a"].view(np.float32).reshape(n, m, 4)
                assert np.array_equal(la.view(np.uint32), d_labels.cpu().numpy().view(np.uint32)), "host != device call"
                vis_a, vis_c = la[..., 3] > 0, host["c"][..., 3] > 0
                row["visible_per_view"] = float(vis_a.sum()) / n
                row["c_equal_visibility_share"] = float((vis_a == vis_c).mean())
                row["label_bytes_per_call"] = n * m * 16
                results["%s_%d" % (vname, m)] = row
    torch.cuda.synchronize()
    line = {"what": "views/s of the labels calls, C2 DEM (synthetic SRTM1, 150 km radius), %dx%d, window -180.05..179.85, %d views "
                    "per call, CUDA events around whole calls" % (W, H, n),
            "gpu": gpu_info(), "results": results}
    text = json.dumps(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


def gpu_info():
    import subprocess
    import torch
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                              "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi name,power.limit,clocks.sm,clocks.max.sm": out}


def C_ctx(h):
    import ctypes
    return ctypes.byref(h.context)


if __name__ == "__main__":
    main()
