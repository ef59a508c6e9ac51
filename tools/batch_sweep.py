"""Batch throughput of the library it loads on the C2 workload:

    python tools/batch_sweep.py [--out sweep.jsonl] [--reps 5] [--batches 16,64]

Per batch size: device-resident panoramas/s for the benchmark viewpoint repeated (what bench.py's `value` is) and for
distinct viewpoints of the 8x8 grid over the central degree (C5 flavour), with the host time spent enqueueing per
panorama.  To compare a compile-time variant, build it under another name (build.py: build_library(extra_flags,
name=...)) and run this once per library with HORIZONATOR_LIBRARY=<path>.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import horizonator_b200 as hz  # noqa: E402
from tools import synth  # noqa: E402

C2_LAT, C2_LON = 34.0 + 1.0 / 7200.0, -117.0 + 1.0 / 7200.0


def grid_views(g=8):
    return [(33.5 + (j + 0.5) / g + 1.0 / 7200.0, -117.5 + (i + 0.5) / g + 1.0 / 7200.0, -180.05, 179.95)
            for j in range(g) for i in range(g)]


def timed(h, views, B, d_img, d_rng, reps):
    st = torch.cuda.current_stream()
    assert st.cuda_stream != 0      # stream 0 would make every call synchronous
    for _ in range(2):
        for k in range(0, len(views), B):
            h.render_batch_device(views[k:k + B], d_img.data_ptr(), d_rng.data_ptr(), st.cuda_stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(st)
    for _ in range(reps):
        for k in range(0, len(views), B):
            h.render_batch_device(views[k:k + B], d_img.data_ptr(), d_rng.data_ptr(), st.cuda_stream)
    e1.record(st)
    host = time.perf_counter() - t0
    torch.cuda.synchronize()
    n = reps * len(views)
    # host time per panorama of a few calls from an idle context (nothing can block on a full ring)
    t0 = time.perf_counter()
    k_free = 0
    for k in range(0, min(len(views), 4 * B), B):
        h.render_batch_device(views[k:k + B], d_img.data_ptr(), d_rng.data_ptr(), st.cuda_stream)
        k_free += len(views[k:k + B])
    host_free = (time.perf_counter() - t0) / k_free * 1e6
    torch.cuda.synchronize()
    return n / (e0.elapsed_time(e1) / 1e3), host_free


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batches", default="16,64")
    ap.add_argument("--once", type=int, default=0, help="for ncu: after two warm-up calls, ONE call of this many "
                    "panoramas of the benchmark viewpoint, nothing else")
    ap.add_argument("--grid", action="store_true", help="with --once: the distinct viewpoints of the 8x8 grid (C5 flavour) "
                    "instead of the benchmark viewpoint repeated")
    ap.add_argument("--grid-size", type=int, default=8, help="distinct viewpoints: a g x g grid over the central degree")
    a = ap.parse_args()
    tiles = synth.config2_tiles(os.environ.get("HZ_BENCH_TILES", "/tmp/hz_tiles_c2"))
    h = hz.horizonator(C2_LAT, C2_LON, 3600, 600, SRTM1=True, dir_dems=tiles, render_radius_m=150000.)
    h.set_zextents(100., 150000.)
    torch.cuda.set_stream(torch.cuda.Stream())
    Bmax = max([int(b) for b in a.batches.split(",")] + [a.once])
    d_img = torch.empty((Bmax, 600, 3600, 3), dtype=torch.uint8, device="cuda")
    d_rng = torch.empty((Bmax, 600, 3600), dtype=torch.float32, device="cuda")
    if a.once:
        g = grid_views(a.grid_size)
        v = (g * (1 + a.once // len(g)))[:a.once] if a.grid else [(C2_LAT, C2_LON, -180.05, 179.95)] * a.once
        for _ in range(3):
            h.render_batch_device(v, d_img.data_ptr(), d_rng.data_ptr(), torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
        return
    grid = grid_views(a.grid_size)
    row = {"library": hz.LIBRARY_PATH}
    for B in (int(b) for b in a.batches.split(",")):
        same, enq_same = timed(h, [(C2_LAT, C2_LON, -180.05, 179.95)] * max(B, 64), B, d_img, d_rng, a.reps)
        dist, enq_dist = timed(h, grid, B, d_img, d_rng, a.reps)
        row["B%d" % B] = {"same_view_pano_s": round(same), "host_us_per_pano": round(enq_same, 2),
                          "grid_pano_s": round(dist), "grid_host_us_per_pano": round(enq_dist, 2)}
    line = json.dumps(row)
    print(line, flush=True)
    if a.out:
        with open(a.out, "a") as out:
            out.write(line + "\n")


if __name__ == "__main__":
    main()
