#!/usr/bin/env python
"""bench.py -- panoramas/s of the render hot path on N B200s (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--batch B] [--dump-outputs DIR]

Workload (N=1 and per rank for N>1): BASELINE.json configs[1] ("C2") -- synthetic SRTM1 tiles N32..N35 x
W119..W116, viewer (34+1/7200, -117+1/7200), render_radius_m = 150 km (R = 5858 cells, 137 M vertices, 274 M
triangles), 3600x600 panorama + range image, az [-180.05, 179.95], znear 100 m, zfar 150 km.  A step is one
call of horizonator_render_batch_device() with --batch (default 256) panoramas per rank on a real CUDA stream: the
library renders them in chunks of up to 64 views, each chunk ONE chain of kernel launches with a view dimension,
chunks alternating between 4 streams.  With N>1 every rank does the same against its own copy of the DEM (weak
scaling, no collective on the data path; NCCL only for the barrier/max of times).

value      device-resident throughput: K steps x batch panoramas / time; outputs stay in HBM, CUDA events on the
           stream the work is queued on, max over ranks
e2e        the same metric through the reference-facing call horizonator_render_offscreen(): one panorama per
           call into (page-locked) HOST buffers, device->host copy inside the timed region; also into pageable
           buffers, through the batch call, and against the box's concurrent device->host ceiling measured in the run
roofline   achieved = algorithmic bytes per panorama (SURVEY 8d: 2*(2R)^2 + 7*W*H) x measured panoramas/s against
           MEASURED_PEAKS.json hbm_gbs; issue = warp instructions per panorama (ncu capture of this configuration,
           profiles/batch_profile.json) x panoramas/s against the SMs' issue peak; per-stage times and the latency of
           a lone panorama
aux        c5_grid: BASELINE configs[4], the 64x64 grid of DISTINCT viewpoints, each rank its own rows;
           lone_ms_special_views: eye 3/12 km up, zoomed-in windows; c3_sweep: configs[2], Python render() pan/zoom
           sweep through the reference's own compiled binding and through the ctypes mirror; c4_wedge (N > 1):
           configs[3], one 36000x4000 panorama by azimuth wedge, assembled in device memory (peer stores over NVLink)
           and in one shared host buffer (every rank over its own PCIe link)
cpu_baseline  the unmodified reference on Mesa llvmpipe on the host cores (rank 0, N=1): one steady-state frame

--impl reference: the reference's own horizonator-lib.c + dem.c + GLSL (compiled unmodified, oracle/_ref) rendering
the same workload on the host cores on Mesa llvmpipe (fallback: on the oracle's software-GL restatement).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C2 = dict(lat=34.0 + 1.0 / 7200.0, lon=-117.0 + 1.0 / 7200.0, W=3600, H=600, radius_m=150000.0,
          az0=-180.05, az1=179.95, znear=100.0, zfar=150000.0, R=5858)
TILES_DIR = os.environ.get("HZ_BENCH_TILES", "/tmp/hz_tiles_c2")


def algorithmic_bytes(R, W, H):
    return 2 * (2 * R) ** 2 + 7 * W * H          # SURVEY.md 8(d)


DUMP_SAMPLE = 1 << 19           # pixels drawn from the whole step for the *_sample arrays of --dump-outputs


def dump_outputs(directory, d_img, d_rng):
    """--dump-outputs: what one batch call handed back (d_img (B, H, W, 3) uint8 B,G,R, d_rng (B, H, W) float32), as
    .npy files that two builds can be compared by, 47 MB for the C2 workload:
      image.npy (H, W, 3), ranges.npy (H, W)            the step's first panorama in full, float32
      sample_index.npy (N,)                             flat indices into (B, H, W), seed 0, sorted, float64
      image_sample.npy (N, 3), ranges_sample.npy (N,)   those pixels of every panorama of the step, float32"""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    B, H, W = d_rng.shape
    n = B * H * W
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(DUMP_SAMPLE, n), replace=False))
    d_idx = torch.from_numpy(idx).to(d_rng.device)
    out = {"image": d_img[0].float(), "ranges": d_rng[0],
           "sample_index": torch.from_numpy(idx.astype(np.float64)),
           "image_sample": d_img.view(n, 3)[d_idx].float(), "ranges_sample": d_rng.view(n)[d_idx]}
    for name, t in out.items():
        np.save(os.path.join(directory, name + ".npy"), t.cpu().numpy())


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + clock-event (throttle) reasons sampled DURING the timed region: NVML polled every ~2 ms from a
    thread (the region can be shorter than nvidia-smi's sampling period); nvidia-smi -lms as the fallback
    (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.samples = []          # (time, sm_mhz, sm_max_mhz, set of reasons)
        self.stop_flag = False
        self.thread = None
        self.how = None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.gpu])
            except (ValueError, IndexError):
                pass
        return self.gpu

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            hnd = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            smmax = float(pynvml.nvmlDeviceGetMaxClockInfo(hnd, pynvml.NVML_CLOCK_SM))
            names = (("hw_slowdown", pynvml.nvmlClocksEventReasonHwSlowdown),
                     ("hw_thermal_slowdown", pynvml.nvmlClocksEventReasonHwThermalSlowdown),
                     ("sw_thermal_slowdown", pynvml.nvmlClocksEventReasonSwThermalSlowdown),
                     ("sw_power_cap", pynvml.nvmlClocksEventReasonSwPowerCap))

            def poll():
                while not self.stop_flag:
                    try:
                        mhz = float(pynvml.nvmlDeviceGetClockInfo(hnd, pynvml.NVML_CLOCK_SM))
                        bits = pynvml.nvmlDeviceGetCurrentClocksEventReasons(hnd)
                        self.samples.append((time.time(), mhz, smmax, {n for n, b in names if bits & b}))
                    except Exception:
                        pass
                    time.sleep(0.002)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            self.how = "nvml"
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self._physical_index()), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
            self.how = "nvidia-smi"
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                mhz, smmax = float(f[1]), float(f[2])
            except ValueError:
                continue
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            self.samples.append((time.time(), mhz, smmax,
                                 {n for n, v in zip(names, f[5:9]) if v.lower().startswith("active")}))

    def stop(self, t0, t1):
        if self.how is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML and no nvidia-smi"]}
        self.stop_flag = True
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
        elif self.thread is not None:
            self.thread.join(timeout=1.0)
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples in the timed region"], "how": self.how}
        sm = sorted(s[1] for s in inside)
        reasons = set()
        for s in inside:
            reasons |= s[3]
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": max(s[2] for s in inside),
                "reasons": sorted(reasons), "samples": len(inside), "how": self.how}


def ensure_tiles(rank, barrier):
    from tools import synth
    if rank == 0:
        synth.config2_tiles(TILES_DIR)
    barrier()
    return TILES_DIR


def c5_grid(world, rank, g=64):
    """BASELINE configs[4] ("C5"): the g x g grid of viewpoints over the central degree of the DEM, dealt to the ranks
    by grid row, round-robin (disjoint; 4096 / world viewpoints each; neighbouring rows cost about the same, so the
    ranks get equal work -- contiguous blocks of rows would give each rank a different kind of terrain)."""
    rows = range(rank, g, world)
    return [(33.5 + (j + 0.5) / g + 1.0 / 7200.0, -117.5 + (i + 0.5) / g + 1.0 / 7200.0) for j in rows for i in range(g)]


# ------------------------------------------------------------------------------------------------ our arm

class StdoutToStderr:
    """stdout carries exactly one JSON line.  Libraries print there too (NCCL writes its version banner to file
    descriptor 1 when NCCL_DEBUG=VERSION): while this is active, descriptor 1 points at stderr; restore() puts it
    back right before the line is printed."""

    def __init__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def restore(self):
        if self.saved is not None:
            sys.stdout.flush()
            os.dup2(self.saved, 1)
            os.close(self.saved)
            self.saved = None


def load_reference_binding():
    """The reference's own horizonator-pywrap.c, compiled unmodified against include/ and linked to the product library
    (oracle/Makefile target `pywrap`; prebuilt, travels with the snapshot).  None where it was never built."""
    import glob
    import importlib.util
    so = glob.glob(os.path.join(ROOT, "oracle", "_ref", "pywrap", "horizonator*.so"))
    if not so:
        return None
    try:
        spec = importlib.util.spec_from_file_location("horizonator", so[0])
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    except Exception as e:          # e.g. numpy ABI mismatch
        sys.stderr.write("bench: reference binding not loadable: %r\n" % (e,))
        return None


def c3_sweep(render, n=48):
    """BASELINE configs[2] ("C3"): pan/zoom re-render sweep through a Python render(az0, az1, znear=, zfar=) callable:
    a pan around the circle at 60 degrees field of view, then a zoom from 120 to 2 degrees; per-render latency."""
    import numpy as np
    wins = [(c - 30.0, c + 30.0) for c in np.linspace(-150.0, 150.0, n // 2)]
    wins += [(45.0 - f / 2, 45.0 + f / 2) for f in np.geomspace(120.0, 2.0, n - n // 2)]
    for a0, a1 in wins[:3]:
        render(float(a0), float(a1), znear=C2["znear"], zfar=C2["zfar"])
    lat = []
    for a0, a1 in wins:
        t0 = time.perf_counter()
        img, rng = render(float(a0), float(a1), znear=C2["znear"], zfar=C2["zfar"])
        lat.append((time.perf_counter() - t0) * 1e3)
    lat.sort()
    return {"renders": len(lat), "median_ms": lat[len(lat) // 2], "p90_ms": lat[int(len(lat) * 0.9)], "max_ms": lat[-1],
            "mean_ms": sum(lat) / len(lat)}


def run_b200(args):
    quiet = StdoutToStderr()
    import numpy as np
    import ctypes as C
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the renderer has no CPU path")
    torch.cuda.set_device(local)
    os.environ["HORIZONATOR_DEVICE"] = str(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    tiles = ensure_tiles(rank, barrier)
    import horizonator_b200 as hz

    t_init = time.time()
    h = hz.horizonator(C2["lat"], C2["lon"], C2["W"], C2["H"], SRTM1=True, dir_dems=tiles,
                       render_radius_m=C2["radius_m"])
    t_init = time.time() - t_init
    R = h.context.dems.radius_cells
    W, H = C2["W"], C2["H"]
    h.set_zextents(C2["znear"], C2["zfar"])
    K, Wm = args.steps, args.warmup
    c2_view = (C2["lat"], C2["lon"], C2["az0"], C2["az1"])
    peak, peak_src = measured_peak_gbs()
    alg = algorithmic_bytes(R, W, H)

    B = args.batch                      # panoramas per step: one call of the batch entry point
    # (how the library cuts a call into chunks: spread evenly over its 4 view sets, 8 to 64 views each -- render_batch_common())
    chunk = max(min(-(-B // 4), 64), min(B, 8))
    n_chunks = -(-B // chunk)
    d_img = torch.empty((B, H, W, 3), dtype=torch.uint8, device="cuda")
    d_rng = torch.empty((B, H, W), dtype=torch.float32, device="cuda")
    # a stream of its own: the batch call takes stream NULL -- which is what torch's default stream is -- to mean "the
    # context's stream, and wait for the result"; on a real stream it only enqueues, and successive calls overlap
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)

    def render_dev(views):
        h.render_batch_device(views, d_img.data_ptr(), d_rng.data_ptr(), stream.cuda_stream)

    def lone_ms(view, reps=20):
        for _ in range(3):
            render_dev([view])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            render_dev([view])
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    # ---- latency of one panorama at a time, then the same with CUDA events around every stage and the culling
    # counters switched on
    latency_ms = lone_ms(c2_view, min(K, 50))
    h.profile(True)
    h.profile_read()
    for k in range(20):
        render_dev([c2_view])
    torch.cuda.synchronize()
    prof = h.profile_read()
    h.profile(False)
    stats = h.last_render_stats()
    counters = h.render_counters()

    # ---- device-resident throughput (the metric's configuration): K steps of B panoramas of the C2 viewpoint ----
    step_views = [c2_view] * B
    for k in range(Wm):
        render_dev(step_views)
    torch.cuda.synchronize()
    batch_launches = h.last_render_stats()["launches"]
    # host time to enqueue a step, measured while nothing can block (the parameter rings are 16 deep): a few steps
    # from an idle context
    n_free = min(K, 4)
    t0 = time.perf_counter()
    for k in range(n_free):
        render_dev(step_views)
    host_enqueue_us = (time.perf_counter() - t0) / (n_free * B) * 1e6
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.05)
    barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.time()
    ev0.record(stream)
    for k in range(K):
        render_dev(step_views)
    ev1.record(stream)
    torch.cuda.synchronize()
    barrier()
    wall1 = time.time()
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    ms_total_max = max_over_ranks(ms_total)
    value = world * K * B / (ms_total_max / 1e3)
    if args.dump_outputs and rank == 0:         # before the C5 grid below renders into the same buffers
        dump_outputs(args.dump_outputs, d_img, d_rng)

    # ---- C5: distinct viewpoints of the 64x64 grid, this rank's disjoint block, in calls of B ----
    grid = [(la, lo, C2["az0"], C2["az1"]) for la, lo in c5_grid(world, rank)]
    n_grid = len(grid) if args.grid_views <= 0 else min(len(grid), args.grid_views)
    grid = grid[:n_grid]
    for k in range(0, min(n_grid, 2 * B), B):
        render_dev(grid[k:k + B])
    barrier()
    torch.cuda.synchronize()
    ev0.record(stream)
    for k in range(0, n_grid, B):
        render_dev(grid[k:k + B])
    ev1.record(stream)
    torch.cuda.synchronize()
    grid_ms = max_over_ranks(ev0.elapsed_time(ev1))
    n_grid_all = int(max_over_ranks(float(n_grid)))        # (the same on every rank)
    grid_value = world * n_grid_all / (grid_ms / 1e3)
    sample = grid[:: max(1, n_grid // 16)][:16]
    lone = sorted(lone_ms(v, 5) for v in sample)
    hit = []
    for v in sample[:4]:
        render_dev([v])
        torch.cuda.synchronize()
        hit.append(float((d_rng[0] > 0).float().mean().item()))

    # ---- expensive views: the eye high above the terrain, zoomed-in windows ----
    special = {"eye_3km": c2_view + (3000.0,), "eye_12km": c2_view + (12000.0,),
               "zoom_30deg": (C2["lat"], C2["lon"], 30.0, 60.0), "zoom_10deg": (C2["lat"], C2["lon"], 40.0, 50.0),
               "zoom_5deg": (C2["lat"], C2["lon"], 42.5, 47.5)}
    special_ms = {k: lone_ms(v, 5) for k, v in special.items()}

    # ---- end to end through the reference-facing call, host buffers ----
    # host result buffers: page-locked (horizonator_host_alloc), reused across steps
    img = hz.pinned_array((H, W, 3), np.uint8)
    rng = hz.pinned_array((H, W), np.float32)
    ctx = C.byref(h.context)

    def e2e_step(la, lo, img, rng):
        # what horizonator-pywrap.c's render() does per call, minus the numpy allocation
        assert hz.lib.horizonator_pan_zoom(ctx, C2["az0"], C2["az1"])
        assert hz.lib.horizonator_move(ctx, None, la, lo)
        assert hz.lib.horizonator_set_zextents(ctx, C2["znear"], C2["zfar"], C2["znear"], C2["zfar"])
        assert hz.lib.horizonator_render_offscreen(ctx, img.ctypes.data, rng.ctypes.data)

    def e2e_rate(img, rng):
        for k in range(Wm):
            e2e_step(C2["lat"], C2["lon"], img, rng)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(K):
            e2e_step(C2["lat"], C2["lon"], img, rng)
        torch.cuda.synchronize()
        return world * K / max_over_ranks(time.perf_counter() - t0)

    e2e_value = e2e_rate(img, rng)
    hit_fraction = float((rng > 0).mean())
    # same call into ordinary pageable numpy arrays (what an unmodified caller of the reference passes)
    img_p = np.zeros((H, W, 3), np.uint8)
    rng_p = np.zeros((H, W), np.float32)
    e2e_pageable = e2e_rate(img_p, rng_p)
    same_pageable = bool(np.array_equal(img_p, img) and np.array_equal(rng_p, rng))

    # how fast this box moves 7*W*H bytes per panorama from every GPU to page-locked host memory at once, with no
    # rendering at all: the ceiling of any end-to-end number at this number of GPUs
    d_flat = torch.empty((7 * W * H,), dtype=torch.uint8, device="cuda")
    h_flat = torch.empty((7 * W * H,), dtype=torch.uint8).pin_memory()
    for k in range(3):
        h_flat.copy_(d_flat, non_blocking=True)
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(K):
        h_flat.copy_(d_flat, non_blocking=True)
    torch.cuda.synchronize()
    d2h_ceiling = world * K / max_over_ranks(time.perf_counter() - t0)
    del d_flat, h_flat

    # the additive host-pointer batch call: renders and device->host copies of different views overlap
    Bh = min(B, 64)
    bimg = hz.pinned_array((Bh, H, W, 3), np.uint8)
    brng = hz.pinned_array((Bh, H, W), np.float32)
    varr = h._views([c2_view] * Bh)
    for k in range(2):
        assert hz.lib.horizonator_render_batch(ctx, Bh, varr, bimg.ctypes.data, brng.ctypes.data)
    n_b = max(3, K // Bh)
    barrier()
    t0 = time.perf_counter()
    for k in range(n_b):
        assert hz.lib.horizonator_render_batch(ctx, Bh, varr, bimg.ctypes.data, brng.ctypes.data)
    e2e_batch = world * n_b * Bh / max_over_ranks(time.perf_counter() - t0)
    del bimg, brng

    # ---- C3: Python render() pan/zoom sweep -- through the reference's own compiled binding (fresh pageable numpy
    # arrays per call, as it allocates them) and through the ctypes mirror (pooled page-locked arrays) ----
    c3 = None
    if rank == 0:
        c3 = {"mirror": c3_sweep(h.render)}
        ref_binding = load_reference_binding()
        if ref_binding is not None:
            hb = ref_binding.horizonator(C2["lat"], C2["lon"], W, H, SRTM1=True, dir_dems=tiles,
                                         render_radius_m=C2["radius_m"])
            c3["reference_binding"] = c3_sweep(hb.render)
            del hb
        else:
            c3["reference_binding"] = None

    # ---- C4 (N > 1): one 36000 x 4000 panorama by azimuth wedge over the ranks ----
    c4 = c4_wedges(hz, tiles, world, rank, barrier, max_over_ranks) if world > 1 and not args.no_c4 else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    stages = {"prepare": "k_prepare", "near": "k_near+k_raster", "big_near": "k_big",
              "march": "bands: (k_tiles, k_blocks, k_mesh, k_raster) x 2", "big_far": "k_big", "resolve": "k_resolve"}
    # achieved: algorithmic bytes per panorama x panoramas/s of the whole device-resident job (kernels of
    # concurrent panoramas overlap, so a single kernel's duration no longer measures the machine)
    per_gpu = value / world
    achieved = alg * per_gpu / 1e9
    prof_batch = batch_profile()
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    issue_peak = 148 * 4 * sm_mhz * 1e6

    def frac_of_roof(ms):
        return alg / (ms / 1e3) / 1e9 / peak

    mosaic_ms = h.time_mosaic(5)
    out = {
        "metric": "panoramas/sec (SRTM1, 3600x600 px)",
        "value": value, "unit": "panoramas/s",
        "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms_total_max / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": "BASELINE configs[1]: single viewpoint per GPU, synthetic SRTM1 4x4 tiles, 150 km radius "
                        "(R=%d cells, %d triangles), 3600x600 panorama + range image" % (R, h.context.Ntriangles),
            "az_deg": [C2["az0"], C2["az1"]], "znear_m": C2["znear"], "zfar_m": C2["zfar"],
            "panoramas_per_step_per_gpu": B,
            "concurrency": "a step is one horizonator_render_batch_device() call of %d panoramas: %d chunks of %d views, "
                           "each chunk ONE chain of kernel launches with a view dimension (one parameter copy + one CUDA "
                           "graph launch per chunk), chunks alternating between 4 streams; same viewpoint, nothing "
                           "cached between views; distinct viewpoints: see aux.c5_grid" % (B, n_chunks, chunk),
            "l2": "no explicit flush; inputs larger than L2: the int16 DEM square is %.0f MB and its culling pyramid "
                  "%.0f MB, and the panoramas in flight cycle up to 64 visibility buffers of %.0f MB each through the 126 MB "
                  "L2 (hierarchical culling makes one panorama touch only a few tens of MB of the DEM, see "
                  "roofline.traffic)" % (2 * (2 * R) ** 2 / 1e6, 4 * ((2 * R) // 4) ** 2 / 1e6, 8 * W * H / 1e6),
            "parallelism": "viewpoint batch, %d panoramas per GPU per step, DEM replicated, no data-path collective" % B,
        },
        "e2e": {"value": e2e_value, "unit": "panoramas/s",
                "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 7 * W * H,
                "note": "horizonator_pan_zoom+move+set_zextents+render_offscreen into page-locked host buffers; "
                        "per-step inputs are 7 scalars passed as kernel arguments (no H2D copy), outputs 7*W*H "
                        "bytes D2H; one panorama per call, calls back to back",
                "pageable_host_buffers_value": e2e_pageable, "pageable_equals_pinned": same_pageable,
                "batch_call_value": e2e_batch,
                "batch_call_note": "horizonator_render_batch() (additive API): %d views per call into page-locked host "
                                   "memory, copies overlapping the next views' kernels" % Bh,
                "d2h_ceiling_value": d2h_ceiling, "fraction_of_d2h_ceiling": e2e_value / d2h_ceiling,
                "batch_call_fraction_of_d2h_ceiling": e2e_batch / d2h_ceiling,
                "d2h_ceiling_note": "panoramas/s at which %d GPU(s) of this box move 7*W*H bytes each to page-locked host "
                                    "memory concurrently with nothing else going on (plain cudaMemcpyAsync, measured "
                                    "in this run)" % world},
        "gpu_launches": K * n_chunks * batch_launches,
        "roofline": {"bound": "hbm", "kernel": "whole panorama: a chain of %d kernels per chunk of up to 64 views, replayed as "
                               "one CUDA graph (k_prepare, k_near, k_raster, k_big, 10 x (k_tiles, k_blocks_mid, k_mesh, "
                               "k_raster), k_big, k_resolve4)" % batch_launches,
                     "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": (prof_batch or {}).get("dram_bytes_per_panorama"),
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg,
                     "stage_ms_single_panorama": {"%s [%s]" % (k, stages[k]): prof[k] for k in stages},
                     "latency_ms_single_panorama": latency_ms,
                     "frac_single_panorama": frac_of_roof(latency_ms),
                     # the resource that actually binds in batch mode: instruction issue.  Instructions per panorama
                     # from an ncu capture of THIS configuration (profiles/batch_profile.json); peak = SMs x 4 schedulers x SM clock
                     "issue": None if prof_batch is None else {
                         "warp_instructions_per_panorama": prof_batch["warp_instructions_per_panorama"],
                         "peak_warp_instructions_per_s": issue_peak,
                         "frac": per_gpu * prof_batch["warp_instructions_per_panorama"] / issue_peak,
                         "source": prof_batch["source"]},
                     "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum over the kernels of one batched chain "
                                     "divided by its views, from the ncu launch list named in issue.source",
                     "note": "achieved = algorithmic bytes per panorama (one read of the int16 DEM square + one write of "
                             "image and range, SURVEY 8d) x measured panoramas/s over the whole timed region.  Hierarchical "
                             "culling makes the kernels read far less DRAM than the algorithmic figure (see traffic): HBM "
                             "is not what binds, instruction issue is (see issue)"},
        "clocks": clocks,
        "aux": {"init_s": t_init, "mosaic_decode_ms": mosaic_ms,
                "mosaic_decode_gbs": 4 * (2 * R) ** 2 / (mosaic_ms / 1e3) / 1e9,
                "triangles_rasterised": stats["triangles_rasterised"], "big_entries": stats["big_entries"],
                "terrain_pixel_fraction": hit_fraction, "culling": counters,
                "host_enqueue_us_per_panorama": host_enqueue_us,
                "host_enqueue_fraction_of_device_period": host_enqueue_us / (1e6 / per_gpu),
                "host_enqueue_note": "host time of %d back-to-back batch calls from an idle context (nothing to wait "
                                     "for), per panorama; device period = 1/value per GPU" % n_free,
                "c5_grid": {"value": grid_value, "unit": "panoramas/s", "viewpoints_per_gpu": n_grid_all,
                            "what": "BASELINE configs[4]: DISTINCT viewpoints of the 64x64 grid over the central degree "
                                    "(33.5..34.5 N, 117.5..116.5 W), eye 1 m above the local terrain, full circle; "
                                    "each rank renders its own rows of the grid (rows rank, rank + N, ...) in calls of %d" % B,
                            "ratio_to_single_viewpoint_value": grid_value / value,
                            "roofline_frac": alg * (grid_value / world) / 1e9 / peak,
                            "lone_ms": {"min": lone[0], "median": lone[len(lone) // 2], "max": lone[-1], "n": len(lone),
                                        "roofline_frac_min_median_max": [frac_of_roof(lone[-1]), frac_of_roof(lone[len(lone) // 2]),
                                                                         frac_of_roof(lone[0])],
                                        "max_over_c2_view": lone[-1] / latency_ms},
                            "terrain_pixel_fraction_sample": hit},
                "lone_ms_special_views": dict(special_ms, note="device time of one panorama at a time; eye_*: explicit "
                                              "viewer_z above sea level over the C2 position (full circle); zoom_*: azimuth "
                                              "window of that width around 45 degrees"),
                "c3_sweep": c3, "c4_wedge": c4},
    }
    if world == 1 and not args.no_cpu_baseline:
        port = cpu_baseline(tiles, use_ref=False, steps=3)
        real = llvmpipe_baseline()
        out["cpu_baseline"] = real or port
        if real:
            out["cpu_baseline_port"] = port
    quiet.restore()
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def batch_profile():
    """Instructions and DRAM bytes per panorama of the batch configuration, from the committed ncu launch list of
    `tools/batch_sweep.py --once 16` (profiles/README.md says how it was taken)."""
    p = os.path.join(ROOT, "profiles", "batch_profile.json")
    try:
        return json.load(open(p))
    except Exception:
        return None


def c4_wedges(hz, tiles, world, rank, barrier, max_over_ranks):
    """BASELINE configs[3]: one 36000 x 4000 full-circle panorama split by azimuth wedge over the ranks, assembled
    (a) in every rank's device memory by the resolve kernel's peer stores over NVLink, (b) in ONE host buffer that all
    ranks share, each rank copying its own wedge over its own PCIe link; against one GPU doing the whole panorama."""
    import torch
    from horizonator_b200 import sharding
    W, H = 36000, 4000
    try:
        h = hz.horizonator(C2["lat"], C2["lon"], W, H, SRTM1=True, dir_dems=tiles, render_radius_m=C2["radius_m"])
        h.set_zextents(C2["znear"], C2["zfar"])
        h.pan_zoom(-180.0 + 180.0 / W, 180.0 - 180.0 / W)
        h.move(C2["lat"], C2["lon"])
        n = 3

        def timed(fn):
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            barrier()
            t0 = time.perf_counter()
            for _ in range(n):
                fn()
            torch.cuda.synchronize()
            return max_over_ranks((time.perf_counter() - t0) / n * 1e3)

        pp = sharding.PeerPanorama(h)
        peer_ms = timed(lambda: pp.render())
        peer_ck = int(pp.image.sum(dtype=torch.int64).item()), float(pp.ranges.double().sum().item())
        timeouts = pp.timeouts()
        pp.close()
        hp = sharding.HostPanorama(h)
        host_ms = timed(lambda: hp.render())
        barrier()
        host_ck = (int(hp.image.astype("int64").sum()), float(hp.ranges.astype("float64").sum())) if rank == 0 else None
        # one GPU doing all of it: device-resident, and delivered to the same host buffer
        whole_dev_ms = whole_host_ms = None
        whole_ck = None
        if rank == 0:
            fi = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda")
            fr = torch.empty((H, W), dtype=torch.float32, device="cuda")
            st = torch.cuda.current_stream().cuda_stream
            for _ in range(2):
                h.render_wedge_device(0, W, fi.data_ptr(), fr.data_ptr(), st)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n):
                h.render_wedge_device(0, W, fi.data_ptr(), fr.data_ptr(), st)
            torch.cuda.synchronize()
            whole_dev_ms = (time.perf_counter() - t0) / n * 1e3
            whole_ck = int(fi.sum(dtype=torch.int64).item()), float(fr.double().sum().item())
            del fi, fr
            hp.render_whole()
            t0 = time.perf_counter()
            for _ in range(n):
                hp.render_whole()
            whole_host_ms = (time.perf_counter() - t0) / n * 1e3
        barrier()
        hp.close()
        del h
        if rank != 0:
            return None
        return {"what": "BASELINE configs[3]: 36000x4000 full circle, C2 DEM, one azimuth wedge per rank",
                "peer_store_ms_per_panorama": peer_ms, "peer_barrier_timeouts": timeouts,
                "host_delivered_ms_per_panorama": host_ms,
                "one_gpu_device_resident_ms": whole_dev_ms, "one_gpu_host_delivered_ms": whole_host_ms,
                "speedup_host_delivered": whole_host_ms / host_ms, "speedup_device_resident": whole_dev_ms / peer_ms,
                "checksums_equal": bool(peer_ck == whole_ck and host_ck == whole_ck), "checksum": list(whole_ck),
                "bytes_per_panorama": 7 * W * H}
    except Exception as e:      # the headline numbers must survive a failure here
        import traceback
        traceback.print_exc()
        return {"error": repr(e)}


# ------------------------------------------------------------------------------------------------ CPU legs

def cpu_baseline(tiles, use_ref, steps=1, warmup=0, budget_s=25.0):
    """Times the CPU oracle (or the reference build) on the C2 workload with all host threads.
    Bounded: renders are timed until `steps` are done or the budget is spent."""
    from oracle import binding
    cores = os.cpu_count() or 1
    cls = binding.Reference if use_ref else binding.Oracle
    o = cls(C2["lat"], C2["lon"], C2["W"], C2["H"], SRTM1=True, dir_dems=tiles,
            render_radius_m=C2["radius_m"], threads=cores)
    for _ in range(warmup):
        o.render(C2["az0"], C2["az1"], znear=C2["znear"], zfar=C2["zfar"])
    times = []
    t_start = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        o.render(C2["az0"], C2["az1"], znear=C2["znear"], zfar=C2["zfar"])
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s:
            break
    mean = sum(times) / len(times)
    return {"value": 1.0 / mean, "unit": "panoramas/s", "cores": cores,
            "kind": "reference" if use_ref else "port",
            "sample": "%d full C2 panorama(s) (3600x600, 274 M triangles), steady state (DEM loaded), %.2f s each; "
                      "%s, OpenMP over %d threads" %
                      (len(times), mean,
                       "reference horizonator-lib.c+dem.c unmodified on the software-GL restatement (oracle/_ref)"
                       if use_ref else "CPU restatement of the reference GL path (oracle/)", cores),
            "ms_per_render": mean * 1e3}


def _timed_renders(o, steps, warmup, budget_s):
    """warm-up renders (at most a quarter of the budget), then up to `steps` timed ones until the budget is spent"""
    t_begin = time.perf_counter()
    done_w = 0
    for _ in range(warmup):
        o.render(C2["az0"], C2["az1"], znear=C2["znear"], zfar=C2["zfar"])
        done_w += 1
        if time.perf_counter() - t_begin > budget_s / 4:
            break
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        o.render(C2["az0"], C2["az1"], znear=C2["znear"], zfar=C2["zfar"])
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_begin > budget_s:
            break
    return times, done_w


def llvmpipe_child(args):
    """Child process of the reference arm: the reference's horizonator-lib.c + dem.c, unmodified, on Mesa llvmpipe
    (oracle/_ref/libhorizonator_mesa.so).  Own process because a GL driver owns process-wide state (JIT, thread pool)
    and because the parent must survive whatever the driver does.  Prints one JSON line."""
    from oracle import binding
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    o = binding.MesaReference(C2["lat"], C2["lon"], C2["W"], C2["H"], SRTM1=True, dir_dems=TILES_DIR,
                              render_radius_m=C2["radius_m"], threads=cores)
    init_s = time.perf_counter() - t0
    version, renderer = o.gl_strings()
    times, done_w = _timed_renders(o, args.steps, args.warmup, float(os.environ.get("HZ_REF_BUDGET_S", "120")))
    print("LLVMPIPE " + json.dumps({"times": times, "warmup": done_w, "gl_version": version, "gl_renderer": renderer,
                                    "init_s": init_s, "lp_threads": min(cores, 16)}), flush=True)


def _llvmpipe_run(steps, warmup, budget_s):
    """The llvmpipe child process; returns its report or None (stderr says why)."""
    import subprocess
    from oracle import binding
    if not binding.have_mesa() or os.environ.get("HZ_REF_GL", "llvmpipe") != "llvmpipe":
        return None
    try:
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--llvmpipe-child",
                            "--steps", str(steps), "--warmup", str(warmup)],
                           env=dict(os.environ, HZ_REF_BUDGET_S=str(budget_s)),
                           capture_output=True, text=True, timeout=2.5 * budget_s + 300)
        lines = [l for l in p.stdout.splitlines() if l.startswith("LLVMPIPE ")]
        if p.returncode == 0 and lines:
            return json.loads(lines[-1][len("LLVMPIPE "):])
        sys.stderr.write("bench: llvmpipe child failed (rc %d): %s\n" % (p.returncode, p.stderr[-1000:]))
    except Exception as e:      # timeout, missing interpreter, ...
        sys.stderr.write("bench: llvmpipe child failed: %r\n" % (e,))
    return None


def llvmpipe_baseline():
    """cpu_baseline of the B200 arm: one full benchmark panorama in steady state (the frame after a warm-up frame, like
    the reference arm times them: the first frame after init also pays for llvmpipe's shader compilation) by the
    unmodified reference on Mesa llvmpipe on this box's host cores (~2 x 30 s of CPU work), or None where that build
    is absent."""
    r = _llvmpipe_run(steps=1, warmup=1, budget_s=200.0)
    if r is None or not r["times"]:
        return None
    cores = os.cpu_count() or 1
    t = r["times"][0]
    return {"value": 1.0 / t, "unit": "panoramas/s", "cores": cores, "kind": "reference",
            "sample": "1 full C2 panorama (3600x600, 274 M triangles), steady state (second frame after init), %.1f s; the reference's "
                      "horizonator-lib.c + dem.c + GLSL shaders compiled UNMODIFIED on a real OpenGL driver: %s, %s "
                      "(oracle/_ref/libhorizonator_mesa.so); llvmpipe rasterises on %d threads, its vertex and geometry "
                      "stages run on one" % (t, r["gl_renderer"], r["gl_version"], r["lp_threads"]),
            "ms_per_render": t * 1e3}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from tools import synth
    from oracle import binding
    synth.config2_tiles(TILES_DIR)
    if not os.path.exists(binding.ORACLE_SO):
        binding.build(ref=False)
    cores = os.cpu_count() or 1
    budget = float(os.environ.get("HZ_REF_BUDGET_S", "120"))

    # (1) the real thing (north_star: "the reference llvmpipe render timed on the box's host cores"): the unmodified
    #     reference on Mesa llvmpipe, in a child process
    llvmpipe = _llvmpipe_run(args.steps, args.warmup, budget)

    # (2) the same reference sources on the software-GL restatement (oracle/_ref), or the oracle port where the
    #     reference was never compiled: the whole arm when (1) is unavailable, a short second opinion when it is not
    use_ref = binding.have_ref()
    cls = binding.Reference if use_ref else binding.Oracle
    o = cls(C2["lat"], C2["lon"], C2["W"], C2["H"], SRTM1=True, dir_dems=TILES_DIR,
            render_radius_m=C2["radius_m"], threads=cores)
    if llvmpipe is None:
        times_r, done_w_r = _timed_renders(o, args.steps, args.warmup, budget)
    else:
        times_r, done_w_r = _timed_renders(o, min(args.steps, 3), 1, 20.0)
    mean_r = sum(times_r) / len(times_r)
    what_r = ("the reference's horizonator-lib.c + dem.c compiled unmodified (oracle/_ref) on a software-GL "
              "restatement of the driver (oracle/gl_pipeline.c)" if use_ref
              else "CPU restatement of the reference GL path (oracle/)")
    restated = {"value": 1.0 / mean_r, "unit": "panoramas/s", "cores": cores, "kind": "reference" if use_ref else "port",
                "sample": "%d full C2 panorama(s), %.2f s each; %s; OpenMP over %d host threads" %
                          (len(times_r), mean_r, what_r, cores)}

    if llvmpipe is not None:
        times, done_w = llvmpipe["times"], llvmpipe["warmup"]
        mean = sum(times) / len(times)
        kind = "reference"
        sample = ("%d of the requested %d steps timed (budget %.0f s), each one full C2 panorama (3600x600, R=5858, "
                  "274 M triangles) through horizonator_render_offscreen() into host buffers, %.1f s each; the "
                  "reference's horizonator-lib.c + dem.c compiled UNMODIFIED, running its own GLSL shaders on a real "
                  "OpenGL driver: %s, %s (oracle/_ref/libhorizonator_mesa.so; context on GLX pbuffers, no X server); "
                  "llvmpipe rasterises on %d threads, its vertex and geometry stages run on one; %d host cores; "
                  "1 process regardless of --gpus" %
                  (len(times), args.steps, budget, mean, llvmpipe["gl_renderer"], llvmpipe["gl_version"],
                   llvmpipe["lp_threads"], cores))
    else:
        times, done_w, mean, kind = times_r, done_w_r, mean_r, restated["kind"]
        sample = ("%d of the requested %d steps timed (budget %.0f s), each one full C2 panorama (3600x600, R=5858, "
                  "274 M triangles) into host buffers, %.2f s each; %s (Mesa llvmpipe build not available here); "
                  "OpenMP over %d host threads; 1 process regardless of --gpus" %
                  (len(times), args.steps, budget, mean, what_r, cores))
    value = 1.0 / mean
    out = {
        "impl": "reference",
        "metric": "panoramas/sec (SRTM1, 3600x600 px)",
        "value": value, "unit": "panoramas/s",
        "n_gpus": world, "steps": len(times), "warmup": done_w,
        "ms_per_step": mean * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: single viewpoint, synthetic SRTM1 4x4 tiles, 150 km radius "
                               "(R=5858 cells, 274482450 triangles), 3600x600 panorama + range image",
                   "az_deg": [C2["az0"], C2["az1"]], "znear_m": C2["znear"], "zfar_m": C2["zfar"]},
        "cpu_baseline": {"value": value, "unit": "panoramas/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "panoramas/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if llvmpipe is not None:
        out["gl"] = {"version": llvmpipe["gl_version"], "renderer": llvmpipe["gl_renderer"], "init_s": llvmpipe["init_s"]}
        out["restated_gl"] = restated     # the same sources on the oracle's GL restatement: a much faster CPU rasteriser
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--batch", type=int, default=256, help="panoramas per step (one call of the batch entry point)")
    ap.add_argument("--grid-views", type=int, default=0, help="viewpoints of the C5 grid per GPU (0 = its whole block)")
    ap.add_argument("--no-c4", action="store_true", help="skip the 36000x4000 wedge panorama (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's image and ranges (the first panorama in full and "
                         "a seeded sample of all of them) as DIR/<name>.npy; rank 0 only")
    ap.add_argument("--llvmpipe-child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.llvmpipe_child:
        return llvmpipe_child(args)
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
