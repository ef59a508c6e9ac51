#!/usr/bin/env python
"""viewshed_bench.py -- viewsheds/s of horizonator_viewshed_device() on one B200, one JSON line.

    python tools/viewshed_bench.py [--out profiles/<name>.json] [--min-seconds S] [--heights]

Workload: the C2 DEM of bench.py (synthetic SRTM1 4x4 tiles, 150 km radius: N = 11716, 46 860 rays per view) with
outputs left in HBM:
  bench_b<B>   B = 1, 16, 64, 256 copies of the bench viewpoint per call, masks into device memory (B x 17.2 MB)
  bench_b256_counts  the same 256 views, counts only (the masks go through the chunk scratch)
  c5_grid      BASELINE configs[4]: bench.py's 64x64 grid of distinct viewpoints, 4096 views per call, counts only
with --heights also (horizonator_viewshed_heights_device), in the same JSON line:
  heights_bench_b<B>  B = 1, 16 copies of the bench viewpoint, per-view heights into device memory (B x 549 MB)
  least_bench_b256    256 copies of the bench viewpoint, the least heights only (the walk's atomics go into it)
  least_c5_grid       the 4096 C5 viewpoints, the least heights only
Each is timed with CUDA events around whole calls on one stream after one warm-up call, repeated until at least
--min-seconds have passed.  Ray steps per second come from the steps the definition takes (counted on the host from
the eyes: per ray |target - first column or row beyond the eye| + 1), not from a profiler.  The device name and power
limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402  (C2, c5_grid, the tile directory)


def ray_steps(h, views):
    """Steps of the R2 definition (include/horizonator-batch.h) for the eyes of `views`, summed over their rays."""
    d = h.context.dems
    N = h.size
    f = np.float32
    k = np.arange(N)
    ti = np.concatenate([k, k, np.zeros(N - 2, int), np.full(N - 2, N - 1)]).astype(f)
    tj = np.concatenate([np.zeros(N, int), np.full(N, N - 1), k[1:-1], k[1:-1]]).astype(f)
    total = 0
    for v in views:
        vci = (f(v[1]) - f(d.origin_dem_lon_lat[0])) * f(d.cells_per_deg) - f(d.origin_dem_cellij[0])
        vcj = (f(v[0]) - f(d.origin_dem_lon_lat[1])) * f(d.cells_per_deg) - f(d.origin_dem_cellij[1])
        di, dj = ti - vci, tj - vcj
        xmaj = np.abs(di) >= np.abs(dj)
        va, da, ta = np.where(xmaj, vci, vcj), np.where(xmaj, di, dj), np.where(xmaj, ti, tj)
        a0 = np.where(da > 0, np.floor(va) + 1, np.ceil(va) - 1)
        total += int(np.where(da != 0, np.abs(ta - a0) + 1, 0).sum())
    return total


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return {"device": name, "nvidia_smi": out}


def timed(fn, stream, min_seconds):
    import torch
    fn()                                                    # warm-up: scratch allocation, module load
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps, t0 = 0, time.perf_counter()
    a.record(stream)
    while True:
        # each call is waited for before the next is decided on: queued calls would run on past the time asked for
        fn()
        reps += 1
        b.record(stream)
        b.synchronize()
        if reps >= 3 and time.perf_counter() - t0 > min_seconds:
            break
    return a.elapsed_time(b) / reps, reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    ap.add_argument("--min-seconds", type=float, default=2.0)
    ap.add_argument("--heights", action="store_true", help="also time the viewshed heights calls")
    args = ap.parse_args()

    import torch
    import horizonator_b200 as hz
    from tools import synth
    assert torch.cuda.is_available(), "viewshed_bench measures on the GPU only"
    C2 = bench.C2
    tiles = synth.config2_tiles(bench.TILES_DIR)
    h = hz.horizonator(C2["lat"], C2["lon"], 64, 16, SRTM1=True, dir_dems=tiles, render_radius_m=C2["radius_m"])
    N = h.size
    w32 = (N + 31) // 32
    stream = torch.cuda.Stream()
    s = stream.cuda_stream
    counts = torch.zeros((N, N), dtype=torch.int32, device="cuda")
    masks = torch.empty((256, N, w32), dtype=torch.int32, device="cuda")
    one = [(C2["lat"], C2["lon"])]
    steps_one = ray_steps(h, one)
    results = {}

    def record(name, views, ms, reps, what):
        n = len(views)
        steps = steps_one * n if all(v == one[0] for v in views) else ray_steps(h, views)
        results[name] = {"views": n, "ms_per_call": ms, "calls_timed": reps, "viewsheds_per_s": n / ms * 1e3,
                         "ray_steps_per_view": steps / n, "ray_steps_per_s": steps / ms * 1e3, "outputs": what}
        print(name, json.dumps(results[name]), file=sys.stderr, flush=True)

    with torch.cuda.stream(stream):
        for B in (1, 16, 64, 256):
            views = one * B
            ms, reps = timed(lambda: h.viewshed_device(views, d_masks=masks.data_ptr(), stream=s), stream,
                             args.min_seconds)
            record("bench_b%d" % B, views, ms, reps, "masks in HBM")
        views = one * 256
        ms, reps = timed(lambda: h.viewshed_device(views, d_counts=counts.data_ptr(), stream=s), stream, args.min_seconds)
        record("bench_b256_counts", views, ms, reps, "counts in HBM")
        grid = [(la, lo) for la, lo in bench.c5_grid(1, 0)]
        ms, reps = timed(lambda: h.viewshed_device(grid, d_counts=counts.data_ptr(), stream=s), stream, args.min_seconds)
        record("c5_grid", grid, ms, reps, "counts in HBM")
        if args.heights:
            least = torch.empty((N, N), dtype=torch.float32, device="cuda")
            heights = torch.empty((16, N, N), dtype=torch.float32, device="cuda")
            for B in (1, 16):
                views = one * B
                ms, reps = timed(lambda: h.viewshed_heights_device(views, d_heights=heights.data_ptr(), stream=s),
                                 stream, args.min_seconds)
                record("heights_bench_b%d" % B, views, ms, reps, "per-view heights in HBM")
            del heights
            # each call folds into least filled with +inf (the fill, 0.1 ms, is inside the timed window), as a
            # caller's first call does
            def fold(views):
                least.fill_(float("inf"))
                h.viewshed_heights_device(views, d_least=least.data_ptr(), stream=s)
            views = one * 256
            ms, reps = timed(lambda: fold(views), stream, args.min_seconds)
            record("least_bench_b256", views, ms, reps, "least heights in HBM")
            ms, reps = timed(lambda: fold(grid), stream, args.min_seconds)
            record("least_c5_grid", grid, ms, reps, "least heights in HBM")
    torch.cuda.synchronize()

    line = {"what": "viewsheds/s of horizonator_viewshed_device(), C2 DEM (synthetic SRTM1, 150 km radius, N=%d, "
                    "%d rays per view), outputs in HBM, CUDA events around whole calls" % (N, 4 * N - 4),
            "gpu": gpu_info(), "results": results}
    text = json.dumps(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
