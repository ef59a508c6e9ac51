#!/usr/bin/env python
"""pick_bench.py -- views/s of the ground-point calls (horizonator_pick_batch*) on one B200, one JSON line.

    python tools/pick_bench.py [--out profiles/<name>.json] [--min-seconds S]

Workload: the C2 DEM and image of bench.py (synthetic SRTM1 4x4 tiles, 150 km radius, 3600 x 600, the bench's
full-circle window), 256 views per call, two view sets: `bench` (the bench viewpoint, 256 times) and `c5` (the 4096
viewpoints of bench.py's C5 grid, 256 per call in turn).  Per view set:
  a_host_1000      horizonator_pick_batch: 1 000 random pixels per view into page-locked host memory, no panorama
  b_device_1000    horizonator_pick_batch_device, the same pixels, queries only (no image, no range image)
  c_device_whole   horizonator_pick_batch_device, every pixel (69 MB of ground points per view into HBM)
  d_device_ranges  horizonator_render_batch_device, range images into HBM: the render alone, the ceiling
Each is timed with CUDA events around whole calls on one stream after one warm-up call, repeated until at least
--min-seconds have passed.  k_pick's own device time comes from torch.profiler (CUDA activities) over a few calls of
b and c, in a separate pass.  The card's name, power limit and clocks are read in the same run.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402  (C2, c5_grid, the tile directory)
from tools.annotate_bench import gpu_info  # noqa: E402
from tools.viewshed_bench import timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--min-seconds", type=float, default=2.0)
    args = ap.parse_args()

    import torch
    import horizonator_b200 as hz
    from tools import synth
    assert torch.cuda.is_available(), "pick_bench measures on the GPU only"
    C2 = bench.C2
    tiles = synth.config2_tiles(bench.TILES_DIR)
    W, H = C2["W"], C2["H"]
    h = hz.horizonator(C2["lat"], C2["lon"], W, H, SRTM1=True, dir_dems=tiles, render_radius_m=C2["radius_m"])
    h.set_zextents(C2["znear"], C2["zfar"])
    n, m = 256, 1000
    grid = [(la, lo, C2["az0"], C2["az1"]) for la, lo in bench.c5_grid(1, 0)]
    view_sets = {"bench": [[(C2["lat"], C2["lon"], C2["az0"], C2["az1"])] * n],
                 "c5": [grid[k:k + n] for k in range(0, len(grid), n)]}
    rs = np.random.default_rng(1)
    px = np.stack([rs.integers(0, W, (n, m)), rs.integers(0, H, (n, m))], axis=2).astype(np.int32)
    d_px = torch.as_tensor(px, device="cuda")
    stream = torch.cuda.Stream()
    s = stream.cuda_stream
    d_ranges = torch.empty((n, H, W), dtype=torch.float32, device="cuda")
    d_query = torch.empty((n, m, 32), dtype=torch.uint8, device="cuda")
    d_whole = torch.empty((n, H, W, 32), dtype=torch.uint8, device="cuda")
    results = {}
    with torch.cuda.stream(stream):
        for vname, calls in view_sets.items():
            turn = {"k": 0}

            def views():
                turn["k"] += 1
                return calls[turn["k"] % len(calls)]

            def a():
                h.pick(views(), px)

            def b():
                h.pick_device(views(), d_px, d_query, stream=s)

            def c():
                h.pick_device(views(), None, d_whole, stream=s)

            def d():
                h.render_batch_device(views(), 0, d_ranges.data_ptr(), s)

            row = {}
            for name, fn in (("a_host_1000", a), ("b_device_1000", b), ("c_device_whole", c), ("d_device_ranges", d)):
                turn["k"] = 0
                ms, reps = timed(fn, stream, args.min_seconds)
                row[name] = {"ms_per_call": ms, "calls_timed": reps, "views_per_s": n / ms * 1e3}
                print(vname, name, json.dumps(row[name]), file=sys.stderr, flush=True)
            row["c_store_bytes_per_call"] = n * H * W * 32
            row["c_store_GB_per_s"] = row["c_store_bytes_per_call"] / row["c_device_whole"]["ms_per_call"] / 1e6
            # k_pick's own device time (torch.profiler, CUDA activities), mean per call of b and of c
            from torch.profiler import ProfilerActivity, profile
            for name, fn in (("b", b), ("c", c)):
                turn["k"] = 0
                fn()
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(4):
                        fn()
                    torch.cuda.synchronize()
                ks = [e for e in prof.key_averages() if "k_pick" in e.key]
                tot = sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) for e in ks)
                row["k_pick_ms_per_call_" + name] = tot / 4 / 1e3
            results[vname] = row
    torch.cuda.synchronize()
    line = {"what": "views/s of the ground-point calls, C2 DEM (synthetic SRTM1, 150 km radius), %dx%d, window %g..%g, "
                    "%d views per call, %d pixels per view in the query cases, CUDA events around whole calls"
                    % (W, H, C2["az0"], C2["az1"], n, m),
            "gpu": gpu_info(), "results": results}
    text = json.dumps(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
