#!/usr/bin/env python
"""skyline_bench.py -- views/s of the skyline match calls (horizonator_skyline_match*) on one B200, one JSON line.

    python tools/skyline_bench.py [--out profiles/<name>.json] [--min-seconds S]

Workload: the C2 DEM and image of bench.py (synthetic SRTM1 4x4 tiles, 150 km radius, 3600 x 600, the bench's
full-circle window), 256 views per call, two view sets: `bench` (the bench viewpoint, 256 times) and `c5` (the 4096
viewpoints of bench.py's C5 grid, 256 per call in turn); observed skylines of m = 600 and m = 3600 samples (the bench
view's own skyline from column 1000 on, so that the samples look like a photo's).  Per combination:
  a_host_scores     horizonator_skyline_match: scores into page-locked host memory, no panorama
  b_device_scores   horizonator_skyline_match_device, scores only (no image, no range image)
  c_profile_torch   the same answer the old way: horizonator_render_batch_device range images into HBM,
                    horizonator_horizon_profile_device, then the same rule in torch (samples in chunks of 100)
  d_device_ranges   horizonator_render_batch_device, range images into HBM: the render alone, the ceiling
  rows_only         horizonator_skyline_match_device, skylines only (rows, no scores); b less this
                    (b_minus_rows_ms_per_call) is the part of k_skyline_score's time that the other view sets' renders
                    do not hide
Each is timed with CUDA events around whole calls on one stream after one warm-up call, repeated until at least
--min-seconds have passed.  k_skyline_score's own device time comes from torch.profiler (CUDA activities) over a
few calls of b, in a separate pass.  The card's name, power limit and clocks are read in the same run.
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


def torch_scores(rows, dx, y, clip, wrap, chunk=100):
    """The rule of horizonator-batch.h in torch over (n, W) int32 rows, samples in chunks (their sum order differs from
    the kernel's: equal to the last few float bits)."""
    import torch
    n, W = rows.shape
    h = torch.arange(W, device=rows.device, dtype=torch.int64)
    total = torch.zeros((n, W), dtype=torch.float32, device=rows.device)
    for i0 in range(0, len(dx), chunk):
        c = h[None, :] + dx[i0:i0 + chunk, None]                            # (k, W)
        if wrap:
            c = torch.remainder(c, W)
        missing = (c < 0) | (c >= W)
        s = rows[:, c.clamp(0, W - 1)]                                       # (n, k, W)
        d = torch.fmin(((s.float() - 0.5) - y[None, i0:i0 + chunk, None]).abs(), torch.tensor(clip, device=rows.device))
        d = torch.where(missing[None] | (s < 0), torch.full_like(d, clip), d)
        total += d.sum(dim=1)
    return total / float(len(dx))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--min-seconds", type=float, default=2.0)
    args = ap.parse_args()

    import torch
    import horizonator_b200 as hz
    from tools import synth
    assert torch.cuda.is_available(), "skyline_bench measures on the GPU only"
    C2 = bench.C2
    tiles = synth.config2_tiles(bench.TILES_DIR)
    W, H = C2["W"], C2["H"]
    h = hz.horizonator(C2["lat"], C2["lon"], W, H, SRTM1=True, dir_dems=tiles, render_radius_m=C2["radius_m"])
    h.set_zextents(C2["znear"], C2["zfar"])
    n = 256
    grid = [(la, lo, C2["az0"], C2["az1"]) for la, lo in bench.c5_grid(1, 0)]
    view_sets = {"bench": [[(C2["lat"], C2["lon"], C2["az0"], C2["az1"])] * n],
                 "c5": [grid[k:k + n] for k in range(0, len(grid), n)]}
    own, _ = h.skyline(view_sets["bench"][0][:1])
    clip = 8.0
    stream = torch.cuda.Stream()
    s = stream.cuda_stream
    d_ranges = torch.empty((n, H, W), dtype=torch.float32, device="cuda")
    d_rows = torch.empty((n, W), dtype=torch.int32, device="cuda")
    d_rr = torch.empty((n, W), dtype=torch.float32, device="cuda")
    d_scores = torch.empty((n, W), dtype=torch.float32, device="cuda")
    results = {}
    with torch.cuda.stream(stream):
        for vname, calls in view_sets.items():
            for m in (600, 3600):
                cols = (1000 + np.arange(m)) % W
                smp = np.zeros(m, hz.SKYLINE_SAMPLE_DTYPE)
                smp["dx"] = np.arange(m)
                smp["y"] = own[0, cols] - 0.5
                d_smp = torch.as_tensor(smp.view(np.int32).reshape(-1, 2), device="cuda")
                t_dx = torch.as_tensor(smp["dx"].astype(np.int64), device="cuda")
                t_y = torch.as_tensor(smp["y"], device="cuda")
                turn = {"k": 0}

                def views():
                    turn["k"] += 1
                    return calls[turn["k"] % len(calls)]

                def a():
                    h.skyline_match(views(), smp, clip_rows=clip)

                def b():
                    h.skyline_match_device(views(), d_smp, d_scores, clip_rows=clip, stream=s)

                def b_rows():
                    h.skyline_match_device(views(), d_smp, 0, d_rows, stream=s)

                def c():
                    v = views()
                    h.render_batch_device(v, 0, d_ranges.data_ptr(), s)
                    h.horizon_profile_device(d_ranges.data_ptr(), len(v), d_rows.data_ptr(), d_rr.data_ptr(), s)
                    d_scores.copy_(torch_scores(d_rows, t_dx, t_y, clip, True))

                def d():
                    h.render_batch_device(views(), 0, d_ranges.data_ptr(), s)

                row = {}
                for name, fn in (("a_host_scores", a), ("b_device_scores", b), ("c_profile_torch", c),
                                 ("d_device_ranges", d), ("rows_only", b_rows)):
                    turn["k"] = 0
                    ms, reps = timed(fn, stream, args.min_seconds)
                    row[name] = {"ms_per_call": ms, "calls_timed": reps, "views_per_s": n / ms * 1e3}
                    print(vname, m, name, json.dumps(row[name]), file=sys.stderr, flush=True)
                row["b_minus_rows_ms_per_call"] = row["b_device_scores"]["ms_per_call"] - row["rows_only"]["ms_per_call"]
                # the old route's scores against the kernel's, for the first call's views
                turn["k"] = -1
                b()
                want = d_scores.clone()
                turn["k"] = -1
                c()
                torch.cuda.synchronize()
                row["c_max_abs_diff_to_b"] = float((d_scores - want).abs().max())
                # k_skyline_score's own device time (torch.profiler, CUDA activities), mean per call of b
                from torch.profiler import ProfilerActivity, profile
                turn["k"] = 0
                b()
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(8):
                        b()
                    torch.cuda.synchronize()
                ks = [e for e in prof.key_averages() if "k_skyline_score" in e.key]
                tot = sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) for e in ks)
                row["k_skyline_score_ms_per_call"] = tot / 8 / 1e3
                row["k_skyline_score_launches_per_call"] = sum(e.count for e in ks) / 8
                row["sample_steps_per_call"] = n * W * m
                results["%s_%d" % (vname, m)] = row
    torch.cuda.synchronize()
    line = {"what": "views/s of the skyline match calls, C2 DEM (synthetic SRTM1, 150 km radius), %dx%d, window %g..%g, "
                    "%d views per call, clip_rows %g, wrap, CUDA events around whole calls" % (W, H, C2["az0"], C2["az1"], n, clip),
            "gpu": gpu_info(), "results": results}
    text = json.dumps(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
