"""horizonator_b200 -- B200-native (sm_100a CUDA) renderer behind dkogan/horizonator's interfaces.

The product is the C-ABI shared library ``horizonator_b200/lib/libhorizonator.so`` (headers in
``include/``).  This module is the host-side mirror of the reference's Python binding
(/root/reference/horizonator-pywrap.c): the same type name, constructor arguments, ``render()``
arguments, return values and error behaviour, implemented with ctypes on top of the C ABI.

There is no CPU fallback: importing works anywhere the library file exists, but constructing a
``horizonator`` without a CUDA device raises ``RuntimeError``, and a missing library raises
``ImportError`` at import time.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# HORIZONATOR_LIBRARY: another build of the same library (A/B comparisons of compile-time variants); still in-tree
LIBRARY_PATH = os.environ.get("HORIZONATOR_LIBRARY") or os.path.join(_HERE, "lib", "libhorizonator.so")

HORIZONATOR_ZNEAR_DEFAULT = 100.0   # include/horizonator.h
HORIZONATOR_ZFAR_DEFAULT = 40000.0


class dem_context_t(C.Structure):
    """include/dem.h: horizonator_dem_context_t (352 bytes)."""
    _fields_ = [
        ("dems", (C.c_void_p * 4) * 4),
        ("mmap_sizes", (C.c_size_t * 4) * 4),
        ("mmap_fd", (C.c_int * 4) * 4),
        ("origin_dem_lon_lat", C.c_int * 2),
        ("origin_dem_cellij", C.c_int * 2),
        ("Ndems_ij", C.c_int * 2),
        ("radius_cells", C.c_int),
        ("cells_per_deg", C.c_int),
    ]


class _offscreen_t(C.Structure):
    _fields_ = [
        ("inited", C.c_bool),
        ("frameBufID", C.c_uint32),
        ("renderBufID", C.c_uint32),
        ("depthBufID", C.c_uint32),
        ("width", C.c_int),
        ("height", C.c_int),
    ]


class context_t(C.Structure):
    """include/horizonator.h: horizonator_context_t (472 bytes)."""
    _fields_ = [
        ("Ntriangles", C.c_int),
        ("render_texture", C.c_bool),
        ("use_glut", C.c_bool),
        ("glut_window", C.c_int),
        ("uniforms", C.c_int32 * 17),
        ("program", C.c_uint32),
        ("viewer_lat", C.c_float),
        ("viewer_lon", C.c_float),
        ("dems", dem_context_t),
        ("offscreen", _offscreen_t),
    ]


class view_t(C.Structure):
    """include/horizonator-batch.h: horizonator_view_t."""
    _fields_ = [
        ("lat", C.c_float), ("lon", C.c_float),
        ("viewer_z", C.c_float),
        ("az_deg0", C.c_float), ("az_deg1", C.c_float),
    ]


class poi_t(C.Structure):
    """include/horizonator-batch.h: horizonator_poi_t (24 bytes)."""
    _fields_ = [("lat", C.c_double), ("lon", C.c_double), ("ele", C.c_double)]


class label_t(C.Structure):
    """include/horizonator-batch.h: horizonator_label_t (16 bytes)."""
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("range_m", C.c_float), ("range_rendered_m", C.c_float)]


#: numpy dtype of label_t: what annotate() returns
LABEL_DTYPE = np.dtype([("x", np.float32), ("y", np.float32), ("range_m", np.float32), ("range_rendered_m", np.float32)])


class skyline_sample_t(C.Structure):
    """include/horizonator-batch.h: horizonator_skyline_sample_t (8 bytes)."""
    _fields_ = [("dx", C.c_int32), ("y", C.c_float)]


#: numpy dtype of skyline_sample_t: what skyline_samples() returns
SKYLINE_SAMPLE_DTYPE = np.dtype([("dx", np.int32), ("y", np.float32)])


class pixel_t(C.Structure):
    """include/horizonator-batch.h: horizonator_pixel_t (8 bytes): column, row (0 = top)."""
    _fields_ = [("x", C.c_int32), ("y", C.c_int32)]


class ground_t(C.Structure):
    """include/horizonator-batch.h: horizonator_ground_t (32 bytes)."""
    _fields_ = [("lat", C.c_double), ("lon", C.c_double), ("ele_m", C.c_float), ("range_m", C.c_float),
                ("distance_m", C.c_float), ("triangle", C.c_uint32)]


#: numpy dtype of ground_t: what pick() returns.  Sky: triangle 0xFFFFFFFF, range_m -1, the rest NaN.
GROUND_DTYPE = np.dtype([("lat", np.float64), ("lon", np.float64), ("ele_m", np.float32), ("range_m", np.float32),
                         ("distance_m", np.float32), ("triangle", np.uint32)])


def skyline_samples(rel_az_deg, el_deg, az_width_deg, width, height):
    """An observed skyline given as angles -> its samples (SKYLINE_SAMPLE_DTYPE) for width x height panoramas of windows
    az_width_deg (az_deg1 - az_deg0) wide: points rel_az_deg degrees right of the heading and el_deg above the
    horizontal.  With p = az_width_deg / width degrees per column, dx = rint(rel_az_deg / p) and
    y = (height - 1) / 2 - el_deg / p in double, rounded to float once (horizonator-batch.h)."""
    rel = np.asarray(rel_az_deg, np.float64).ravel()
    el = np.asarray(el_deg, np.float64).ravel()
    p = float(az_width_deg) / width
    out = np.empty(len(rel), SKYLINE_SAMPLE_DTYPE)
    out["dx"] = np.rint(rel / p)
    out["y"] = (height - 1) / 2. - el / p
    return out


def _signatures():
    """{symbol: (restype, argtypes)} of every function include/*.h declares."""
    P = C.POINTER
    ctx = P(context_t)
    f, d, i, b, vp, cp = C.c_float, C.c_double, C.c_int, C.c_bool, C.c_void_p, C.c_char_p
    return {
        "horizonator_init": (b, [ctx, f, f, P(f), i, i, i, f, b, b, b, cp, cp, cp, cp, b]),
        "horizonator_deinit": (None, [ctx]),
        "horizonator_resized": (b, [ctx, i, i]),
        "horizonator_pan_zoom": (b, [ctx, f, f]),
        "horizonator_move": (b, [ctx, P(f), f, f]),
        "horizonator_set_zextents": (b, [ctx, f, f, f, f]),
        "horizonator_redraw": (b, [ctx]),
        "horizonator_pick": (b, [ctx, P(f), P(f), i, i]),
        "horizonator_render_offscreen": (b, [ctx, vp, vp]),
        "horizonator_x_from_az": (b, [P(d), P(d), d, d, d, i]),
        "horizonator_project": (b, [P(d), P(d), P(d), d, d, d, d, d, d, d, d, d, i, i]),
        "horizonator_unproject": (b, [P(f), P(f), i, i, d, d, d, d, d, d, d, i, i]),
        "horizonator_dem_init": (b, [P(dem_context_t), f, f, i, f, cp, b]),
        "horizonator_dem_deinit": (None, [P(dem_context_t)]),
        "horizonator_dem_sample": (C.c_int16, [P(dem_context_t), i, i]),
        "horizonator_dem_bounds_latlon_deg": (None, [P(dem_context_t), P(f), P(f), P(f), P(f)]),
        "horizonator_render_batch_device": (b, [ctx, i, P(view_t), vp, vp, vp]),
        "horizonator_render_batch": (b, [ctx, i, P(view_t), vp, vp]),
        "horizonator_render_wedge_device": (b, [ctx, i, i, vp, vp, vp]),
        "horizonator_download_mosaic": (b, [ctx, vp]),
        "horizonator_time_mosaic": (b, [ctx, i, P(f)]),
        "horizonator_last_render_stats": (b, [ctx, P(C.c_uint * 5)]),
        "horizonator_render_counters": (b, [ctx, P(C.c_uint * 16)]),
        "horizonator_horizon_profile_device": (b, [ctx, vp, i, vp, vp, vp]),
        "horizonator_set_earth_curvature": (b, [ctx, b, f]),
        "horizonator_set_seam_wrap": (b, [ctx, b]),
        "horizonator_set_lod": (b, [ctx, f]),
        "horizonator_peer_alloc": (b, [ctx, C.c_size_t, P(vp), P(C.c_ubyte * 64)]),
        "horizonator_peer_open": (b, [ctx, P(C.c_ubyte * 64), P(vp)]),
        "horizonator_peer_close": (b, [ctx, vp]),
        "horizonator_peer_free": (b, [ctx, vp]),
        "horizonator_render_wedge_peers": (b, [ctx, i, i, i, P(vp), P(vp), vp]),
        "horizonator_peer_barrier": (b, [ctx, i, i, P(vp), C.c_uint, vp]),
        "horizonator_debug_device_math": (b, [i, vp, vp, vp, vp, vp, vp]),
        "horizonator_render_wedge_host": (b, [ctx, i, i, vp, vp]),
        "horizonator_host_register": (b, [vp, C.c_size_t]),
        "horizonator_host_unregister": (b, [vp]),
        "horizonator_host_alloc": (vp, [C.c_size_t]),
        "horizonator_host_free": (None, [vp]),
        "horizonator_profile_enable": (b, [ctx, b]),
        "horizonator_profile_read": (b, [ctx, P(f * 6), P(i)]),
        "horizonator_viewshed_device": (b, [ctx, i, P(view_t), f, vp, vp, vp]),
        "horizonator_viewshed": (b, [ctx, i, P(view_t), f, vp, vp]),
        "horizonator_viewshed_heights_device": (b, [ctx, i, P(view_t), vp, vp, vp]),
        "horizonator_viewshed_heights": (b, [ctx, i, P(view_t), vp, vp]),
        "horizonator_annotate_batch_device": (b, [ctx, i, P(view_t), i, vp, vp, vp, vp, vp]),
        "horizonator_annotate_batch": (b, [ctx, i, P(view_t), i, vp, vp]),
        "horizonator_skyline_match_device": (b, [ctx, i, P(view_t), vp, vp, i, vp, f, b, vp, vp]),
        "horizonator_skyline_match": (b, [ctx, i, P(view_t), vp, vp, i, vp, f, b, vp]),
        "horizonator_pick_batch_device": (b, [ctx, i, P(view_t), i, vp, vp, vp, vp, vp]),
        "horizonator_pick_batch": (b, [ctx, i, P(view_t), i, vp, vp]),
    }


def _declare(lib):
    for name, (res, args) in _signatures().items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise ImportError("%s is stale (no symbol %s): rebuild it with `python horizonator_b200/build.py`"
                              % (LIBRARY_PATH, name)) from None
        fn.restype = res
        fn.argtypes = args
    return lib


#: every symbol include/*.h declares (tests check that the library exports each of them)
EXPORTED_SYMBOLS = tuple(_signatures())

if not os.path.exists(LIBRARY_PATH):
    raise ImportError(
        "%s is missing: build it with `python horizonator_b200/build.py` (needs nvcc). "
        "horizonator_b200 has no CPU fallback." % LIBRARY_PATH)

lib = _declare(C.CDLL(LIBRARY_PATH))


def _enc(s):
    return None if s is None else os.fsencode(s)


def _check(fn, *args):
    """Calls the library function fn; raises RuntimeError("<name>() failed") if it returns false."""
    if not fn(*args):
        raise RuntimeError("%s() failed" % fn.__name__)


class horizonator:
    """SRTM terrain renderer: mirror of the reference's Python type ``horizonator.horizonator``.

    Arguments, defaults and semantics as /root/reference/horizonator-pywrap.c:49-125 and
    horizonator.docstring.  The constructor loads the DEMs around (lat, lon) and is relatively
    slow; ``render()`` is fast.
    """

    def __init__(self, lat, lon, width, height,
                 render_texture=False, SRTM1=False,
                 dir_dems=None, dir_tiles=None, tiles_name=None, tiles_url_fmt=None,
                 allow_downloads=True, render_radius_cells=-1, render_radius_m=-1.):
        self._ctx = context_t()
        if render_radius_cells < 0 and render_radius_m < 0:
            render_radius_cells = 1000                      # pywrap.c:65,98-99
        elif render_radius_cells > 0 and render_radius_m > 0:
            raise RuntimeError("both render_radius_cells,render_radius_m cannot be >0")
        if width < 0 or height < 0:
            raise OverflowError("width, height must be unsigned")   # format "II"
        _check(lib.horizonator_init, C.byref(self._ctx), lat, lon, None,
               int(width), int(height),
               int(render_radius_cells), float(render_radius_m),
               True, bool(render_texture), bool(SRTM1),
               _enc(dir_dems), _enc(dir_tiles), _enc(tiles_name), _enc(tiles_url_fmt),
               bool(allow_downloads))

    def __del__(self):
        ctx = getattr(self, "_ctx", None)
        if ctx is not None and lib is not None:
            lib.horizonator_deinit(C.byref(ctx))

    def close(self):
        lib.horizonator_deinit(C.byref(self._ctx))

    def __str__(self):
        # pywrap.c:133-156: "%.9S" = the first 9 characters of str(float)
        return "Looking out from %s,%s" % (str(float(self._ctx.viewer_lat))[:9], str(float(self._ctx.viewer_lon))[:9])

    # ------------------------------------------------------------------ reference API
    def render(self, az_deg0, az_deg1, lat=-1000., lon=-1000.,
               return_image=True, return_range=True, az_extents_use_pixel_centers=False,
               znear=HORIZONATOR_ZNEAR_DEFAULT, zfar=HORIZONATOR_ZFAR_DEFAULT,
               znear_color=-1., zfar_color=-1.):
        """Mirror of render() at horizonator-pywrap.c:158-279.

        Returns (image, ranges), or just one of them, or () -- image: (H,W,3) uint8 in B,G,R order,
        ranges: (H,W) float32 with -1 where no terrain is seen; top row first.
        """
        if znear_color < 0.:
            znear_color = znear
        if zfar_color < 0.:
            zfar_color = zfar
        if not return_image and not return_range:
            return ()
        W, H = self._ctx.offscreen.width, self._ctx.offscreen.height
        if az_extents_use_pixel_centers:
            az_per_pixel = (az_deg1 - az_deg0) / float(W - 1)
            az_deg0 -= az_per_pixel / 2.
            az_deg1 += az_per_pixel / 2.
        _check(lib.horizonator_pan_zoom, C.byref(self._ctx), az_deg0, az_deg1)
        if lat > -1000.:
            _check(lib.horizonator_move, C.byref(self._ctx), None, lat, lon)
        _check(lib.horizonator_set_zextents, C.byref(self._ctx), znear, zfar, znear_color, zfar_color)
        # fresh arrays per call like the reference (pywrap.c:234-250), but out of a recycling pool of page-locked
        # blocks: the results then arrive by DMA instead of through the driver's pageable staging (3x faster for
        # 15 MB), and a block goes back to the pool when the caller drops the array
        image = _pool.array((H, W, 3), np.uint8) if return_image else None
        ranges = _pool.array((H, W), np.float32) if return_range else None
        _check(lib.horizonator_render_offscreen, C.byref(self._ctx),
               image.ctypes.data if image is not None else None,
               ranges.ctypes.data if ranges is not None else None)
        if return_image and not return_range:
            return image
        if return_range and not return_image:
            return ranges
        return image, ranges

    # ------------------------------------------------------------------ additions (horizonator-batch.h)
    @property
    def width(self):
        return self._ctx.offscreen.width

    @property
    def height(self):
        return self._ctx.offscreen.height

    @property
    def context(self):
        """The underlying horizonator_context_t (ctypes structure)."""
        return self._ctx

    @staticmethod
    def _views(views):
        arr = (view_t * len(views))()
        for k, v in enumerate(views):
            lat, lon, az0, az1 = v[0], v[1], v[2], v[3]
            z = v[4] if len(v) > 4 else -1.
            arr[k] = view_t(lat, lon, z, az0, az1)
        return arr

    def set_zextents(self, znear, zfar, znear_color=-1., zfar_color=-1.):
        if znear_color < 0.:
            znear_color = znear
        if zfar_color < 0.:
            zfar_color = zfar
        _check(lib.horizonator_set_zextents, C.byref(self._ctx), znear, zfar, znear_color, zfar_color)

    def render_batch(self, views, return_image=True, return_range=True):
        """views: sequence of (lat, lon, az_deg0, az_deg1[, viewer_z]).  Host arrays (n,H,W,3), (n,H,W)."""
        n, W, H = len(views), self.width, self.height
        # page-locked blocks from the recycling pool, like render(): the copies of different views then run by DMA and
        # overlap the next views' kernels (into pageable arrays each copy would go through the driver's staging)
        image = _pool.array((n, H, W, 3), np.uint8) if return_image else None
        ranges = _pool.array((n, H, W), np.float32) if return_range else None
        _check(lib.horizonator_render_batch, C.byref(self._ctx), n, self._views(views),
               image.ctypes.data if image is not None else None,
               ranges.ctypes.data if ranges is not None else None)
        return image, ranges

    def render_batch_device(self, views, d_images=0, d_ranges=0, stream=0):
        """Device-pointer variant: d_images / d_ranges are integer device addresses (e.g. tensor.data_ptr()),
        stream an integer cudaStream_t (0 = the context's own stream, synchronous)."""
        _check(lib.horizonator_render_batch_device, C.byref(self._ctx), len(views), self._views(views),
               d_images or None, d_ranges or None, stream or None)

    def render_wedge_device(self, x0, x1, d_image=0, d_ranges=0, stream=0):
        _check(lib.horizonator_render_wedge_device, C.byref(self._ctx), int(x0), int(x1),
               d_image or None, d_ranges or None, stream or None)

    def render_wedge_host(self, x0, x1, image=None, ranges=None):
        """Columns [x0, x1) of the current view into FULL-size host arrays (H,W,3) uint8 / (H,W) float32."""
        _check(lib.horizonator_render_wedge_host, C.byref(self._ctx), int(x0), int(x1),
               image.ctypes.data if image is not None else None,
               ranges.ctypes.data if ranges is not None else None)

    def set_seam_wrap(self, on=True):
        """Opt-in (off by default; the reference drops them): draw triangles across the +-180 degree seam at both
        edges of a full-circle panorama.  See horizonator-batch.h."""
        _check(lib.horizonator_set_seam_wrap, C.byref(self._ctx), bool(on))

    def set_lod(self, max_cell_pixels=0.5):
        """Opt-in level of detail (0 = off, the default; the reference always draws every DEM cell): coarser far mesh
        where a coarser cell still is at most `max_cell_pixels` pixels across.  See horizonator-batch.h."""
        _check(lib.horizonator_set_lod, C.byref(self._ctx), float(max_cell_pixels))

    def set_earth_curvature(self, on=True, refraction=0.13):
        """Opt-in accuracy mode (off by default; the reference is flat-earth): see horizonator-batch.h."""
        _check(lib.horizonator_set_earth_curvature, C.byref(self._ctx), bool(on), float(refraction))

    # peer-memory assembly of wedge-sharded panoramas (horizonator-batch.h); used by sharding.PeerPanorama
    def peer_alloc(self, nbytes):
        """-> (device address, 64-byte handle) of a buffer other ranks can map."""
        ptr, handle = C.c_void_p(), (C.c_ubyte * 64)()
        _check(lib.horizonator_peer_alloc, C.byref(self._ctx), nbytes, C.byref(ptr), C.byref(handle))
        return ptr.value, bytes(handle)

    def peer_open(self, handle):
        ptr = C.c_void_p()
        _check(lib.horizonator_peer_open, C.byref(self._ctx), (C.c_ubyte * 64).from_buffer_copy(handle), C.byref(ptr))
        return ptr.value

    def peer_close(self, ptr):
        lib.horizonator_peer_close(C.byref(self._ctx), ptr)

    def peer_free(self, ptr):
        lib.horizonator_peer_free(C.byref(self._ctx), ptr)

    def peer_barrier(self, rank, d_flags, epoch, stream=0):
        """GPU-side barrier between ranks (horizonator_peer_barrier); d_flags: every rank's flag block address."""
        arr = (C.c_void_p * len(d_flags))(*d_flags)
        _check(lib.horizonator_peer_barrier, C.byref(self._ctx), len(d_flags), int(rank), arr, int(epoch), stream or None)

    def render_wedge_peers(self, x0, x1, d_images, d_ranges, stream=0):
        """d_images / d_ranges: sequences of device addresses of every rank's full image / range buffer (or None)."""
        n = len(d_images) if d_images is not None else len(d_ranges)
        ai = (C.c_void_p * n)(*d_images) if d_images is not None else None
        ar = (C.c_void_p * n)(*d_ranges) if d_ranges is not None else None
        _check(lib.horizonator_render_wedge_peers, C.byref(self._ctx), int(x0), int(x1), n, ai, ar, stream or None)

    def pan_zoom(self, az_deg0, az_deg1):
        _check(lib.horizonator_pan_zoom, C.byref(self._ctx), az_deg0, az_deg1)

    def move(self, lat, lon, viewer_z=None):
        z = C.c_float(-1. if viewer_z is None else viewer_z)
        _check(lib.horizonator_move, C.byref(self._ctx), C.byref(z), lat, lon)
        return z.value

    def mosaic(self):
        """The decoded DEM square as the GPU holds it: (2R, 2R) int16, [j north][i east]."""
        n = 2 * self._ctx.dems.radius_cells
        out = np.empty((n, n), dtype=np.int16)
        _check(lib.horizonator_download_mosaic, C.byref(self._ctx), out.ctypes.data)
        return out

    def time_mosaic(self, reps=10):
        ms = C.c_float(0)
        _check(lib.horizonator_time_mosaic, C.byref(self._ctx), reps, C.byref(ms))
        return ms.value

    def render_into(self, image, ranges):
        """horizonator_render_offscreen() with the current state into caller-owned arrays (either may be
        None): no allocation, and DMA speed when the arrays come from pinned_array()."""
        _check(lib.horizonator_render_offscreen, C.byref(self._ctx),
               image.ctypes.data if image is not None else None,
               ranges.ctypes.data if ranges is not None else None)

    def profile(self, on=True):
        """Record CUDA events around every kernel of every render from now on (see profile_read)."""
        _check(lib.horizonator_profile_enable, C.byref(self._ctx), bool(on))

    def profile_read(self):
        """Mean device ms per render of each kernel since the last read, and the number of renders."""
        ms = (C.c_float * 6)()
        n = C.c_int(0)
        _check(lib.horizonator_profile_read, C.byref(self._ctx), C.byref(ms), C.byref(n))
        return {"prepare": ms[0], "near": ms[1], "big_near": ms[2], "march": ms[3], "big_far": ms[4],
                "resolve": ms[5], "renders": n.value}

    def last_render_stats(self):
        out = (C.c_uint * 5)()
        _check(lib.horizonator_last_render_stats, C.byref(self._ctx), C.byref(out))
        return {"big_entries": out[0], "big_capacity": out[1], "launches": out[2], "device": out[3],
                "triangles_rasterised": out[4]}

    COUNTER_NAMES = ("tiles", "tiles_far", "tiles_window", "tiles_occluded",
                     "blocks", "blocks_far", "blocks_window", "blocks_occluded",
                     "blocks_meshed", "triangles", "big_entries", "occluded_by_grid", "span_blocks")

    def render_counters(self):
        """Culling counters of the most recent render (horizonator_render_counters)."""
        out = (C.c_uint * 16)()
        _check(lib.horizonator_render_counters, C.byref(self._ctx), C.byref(out))
        return dict(zip(self.COUNTER_NAMES, out))

    def horizon_profile_device(self, d_ranges, n, d_rows, d_range, stream=0):
        """Per-column topmost terrain (row, range) of n device range images; all arguments device addresses."""
        _check(lib.horizonator_horizon_profile_device, C.byref(self._ctx), d_ranges, int(n), d_rows, d_range,
               stream or None)

    # viewsheds (horizonator-batch.h: which vertices of the loaded square each view sees)
    @property
    def size(self):
        """N = 2R: the loaded square is N x N vertices."""
        return 2 * self._ctx.dems.radius_cells

    @staticmethod
    def _eyes(views):
        """views: (lat, lon), or (lat, lon, az_deg0, az_deg1[, viewer_z]) as render_batch takes them (the azimuth
        window is ignored: a viewshed covers the full circle)."""
        return horizonator._views([tuple(v) + (0., 0.) if len(v) == 2 else v for v in views])

    def viewshed(self, views, target_height=0., counts=False):
        """Host arrays: masks (n, N, N) bool, [j north][i east], True where the view sees the vertex (a point
        target_height metres above it); with counts=True also (N, N) uint32, how many of the views see each vertex."""
        n, N = len(views), self.size
        w32 = (N + 31) // 32
        words = np.empty((n, N, w32), np.uint32)
        cnt = np.zeros((N, N), np.uint32) if counts else None
        _check(lib.horizonator_viewshed, C.byref(self._ctx), n, self._eyes(views), float(target_height),
               words.ctypes.data, cnt.ctypes.data if counts else None)
        bits = np.unpackbits(words.view(np.uint8), axis=-1, bitorder="little")[..., :N].astype(bool)
        return (bits, cnt) if counts else bits

    def viewshed_device(self, views, d_masks=0, d_counts=0, target_height=0., stream=0):
        """Device-pointer variant: d_masks (n, N, (N+31)//32) uint32 words, overwritten; d_counts (N, N) uint32,
        added to.  Integer device addresses, either may be 0 (not both); stream as render_batch_device."""
        _check(lib.horizonator_viewshed_device, C.byref(self._ctx), len(views), self._eyes(views), float(target_height),
               d_masks or None, d_counts or None, stream or None)

    def viewshed_heights(self, views, least=False):
        """Host arrays: heights (n, N, N) float32, [j north][i east], how far above the ground a point at each vertex
        must rise for the view to see it (+0 where the ground itself is seen, +inf where no ray reaches the vertex);
        with least=True also (N, N) float32, the least of them over the views (horizonator-batch.h)."""
        n, N = len(views), self.size
        h = np.empty((n, N, N), np.float32)
        lst = np.full((N, N), np.inf, np.float32) if least else None
        _check(lib.horizonator_viewshed_heights, C.byref(self._ctx), n, self._eyes(views), h.ctypes.data,
               lst.ctypes.data if least else None)
        return (h, lst) if least else h

    def viewshed_least_height(self, views):
        """(N, N) float32: for every vertex the least height above the ground at which any of the views sees a point
        there -- below it the point stays hidden from all of them.  No per-view array is made."""
        N = self.size
        lst = np.full((N, N), np.inf, np.float32)
        _check(lib.horizonator_viewshed_heights, C.byref(self._ctx), len(views), self._eyes(views), None,
               lst.ctypes.data)
        return lst

    def viewshed_heights_device(self, views, d_heights=0, d_least=0, stream=0):
        """Device-pointer variant: d_heights (n, N, N) float32, overwritten; d_least (N, N) float32, min-folded (fill
        it with +inf first).  Integer device addresses, either may be 0 (not both); stream as render_batch_device."""
        _check(lib.horizonator_viewshed_heights_device, C.byref(self._ctx), len(views), self._eyes(views),
               d_heights or None, d_least or None, stream or None)


    # labels of points of interest (horizonator_annotate_batch*: which POIs each view sees, and where)
    @staticmethod
    def pois_array(pois):
        """A sequence of (lat, lon, ele) or an (m, 3) array -> (m, 3) C-contiguous float64 (horizonator_poi_t[m])."""
        return np.ascontiguousarray(np.asarray(pois, dtype=np.float64).reshape(-1, 3))

    def annotate(self, views, pois):
        """views as render_batch takes them; pois: (lat, lon, ele) each, ele in metres.  Returns an (n, m) structured
        array (LABEL_DTYPE): x, y (marker pixel; all fields -1 where the POI is outside the window), range_m, and
        range_rendered_m (> 0 exactly when the view sees the POI).  Only the labels leave the GPU."""
        p = self.pois_array(pois)
        n, m = len(views), p.shape[0]
        out = _pool.array((n, m, 4), np.float32)
        _check(lib.horizonator_annotate_batch, C.byref(self._ctx), n, self._views(views), m, p.ctypes.data if m else None,
               out.ctypes.data if out.size else None)
        return out.view(LABEL_DTYPE).reshape(n, m)

    def annotate_device(self, views, d_pois, d_labels, d_images=0, d_ranges=0, stream=0, m=None):
        """Device-memory variant.  d_pois: an (m, 3) float64 CUDA tensor, or an integer device address with `m` given;
        d_labels: an (n, m, 4) float32 CUDA tensor (a view as LABEL_DTYPE is the same memory) or an integer address;
        d_images / d_ranges as render_batch_device (0 = not written); stream as render_batch_device."""
        if hasattr(d_pois, "data_ptr"):
            if m is None:
                m = d_pois.shape[0]
            d_pois = d_pois.data_ptr()
        if m is None:
            raise ValueError("annotate_device: m is needed when d_pois is an address")
        if hasattr(d_labels, "data_ptr"):
            d_labels = d_labels.data_ptr()
        _check(lib.horizonator_annotate_batch_device, C.byref(self._ctx), len(views), self._views(views), int(m),
               d_pois or None, d_labels or None, d_images or None, d_ranges or None,
               stream or None)

    # skylines and their match against an observed skyline (horizonator_skyline_match*: where a photo was taken)
    def skyline_samples(self, rel_az_deg, el_deg, az_width_deg):
        """skyline_samples() for this context's W x H panoramas."""
        return skyline_samples(rel_az_deg, el_deg, az_width_deg, self.width, self.height)

    @staticmethod
    def _samples(samples):
        """SKYLINE_SAMPLE_DTYPE array, or a sequence of (dx, y) -> C-contiguous SKYLINE_SAMPLE_DTYPE array."""
        a = np.asarray(samples)
        if a.dtype == SKYLINE_SAMPLE_DTYPE:
            return np.ascontiguousarray(a.ravel())
        a = a.reshape(-1, 2)
        out = np.empty(len(a), SKYLINE_SAMPLE_DTYPE)
        out["dx"], out["y"] = a[:, 0], a[:, 1]
        return out

    def _skyline_call(self, views, samples, clip_rows, wrap, rows, rng, scores):
        n, W = len(views), self.width
        out = {k: _pool.array((n, W), dt) if want else None
               for k, dt, want in (("rows", np.int32, rows), ("range", np.float32, rng), ("scores", np.float32, scores))}
        s = self._samples(samples) if scores else None
        addr = {k: (a.ctypes.data if a is not None and a.size else None) for k, a in out.items()}
        _check(lib.horizonator_skyline_match, C.byref(self._ctx), n, self._views(views), addr["rows"], addr["range"],
               len(s) if scores else 0, s.ctypes.data if scores and len(s) else None, float(clip_rows), bool(wrap),
               addr["scores"])
        return out

    def skyline(self, views):
        """views as render_batch takes them -> (rows (n, W) int32, range (n, W) float32): the topmost terrain pixel of
        each column (image row, 0 = top) and its range, -1 / -1 for an all-sky column.  Only these leave the GPU."""
        out = self._skyline_call(views, None, 1., False, True, True, False)
        return out["rows"], out["range"]

    def skyline_match(self, views, samples, clip_rows=8., wrap=True, rows=False):
        """Scores (n, W) float32 of an observed skyline (samples: skyline_samples(), or (dx, y) pairs) against every
        view at every heading column: the mean error in rows, each sample's clipped at clip_rows (horizonator-batch.h).
        wrap: columns wrap around (full-circle windows).  rows=True: (scores, rows (n, W) int32)."""
        out = self._skyline_call(views, samples, clip_rows, wrap, rows, False, True)
        return (out["scores"], out["rows"]) if rows else out["scores"]

    def skyline_match_device(self, views, d_samples, d_scores=0, d_rows=0, d_range=0, clip_rows=8., wrap=True, stream=0,
                             m=None):
        """Device-memory variant.  d_samples: an (m, 2) int32 CUDA tensor whose rows are (dx, y as float bits), an (m,)
        int64 one, or an integer device address with `m` given; d_scores, d_rows, d_range: (n, W) float32 / int32 /
        float32 CUDA tensors or integer addresses (0 = not written); stream as render_batch_device."""
        if hasattr(d_samples, "data_ptr"):
            if m is None:
                m = d_samples.shape[0]
            d_samples = d_samples.data_ptr()
        if m is None:
            m = 0
        d_scores, d_rows, d_range = (a.data_ptr() if hasattr(a, "data_ptr") else a for a in (d_scores, d_rows, d_range))
        _check(lib.horizonator_skyline_match_device, C.byref(self._ctx), len(views), self._views(views), d_rows or None,
               d_range or None, int(m), d_samples or None, float(clip_rows), bool(wrap), d_scores or None, stream or None)

    def locate(self, views, samples, top=10, clip_rows=8., wrap=True):
        """Where and which way a photo was taken: the `top` best (view index, heading azimuth in degrees, score) of
        skyline_match() over the candidate views and all their headings, best (smallest score) first; ties go to the
        lower view index, then the lower heading column.  The heading of column h is az_deg0 + (h + 0.5) * p."""
        scores = self.skyline_match(views, samples, clip_rows=clip_rows, wrap=wrap)
        W = self.width
        flat = scores.ravel()
        order = np.argsort(flat, kind="stable")[:top]
        out = []
        for i in order:
            k, h = divmod(int(i), W)
            az0, az1 = float(np.float32(views[k][2])), float(np.float32(views[k][3]))
            out.append((k, az0 + (h + 0.5) * (az1 - az0) / W, float(flat[i])))
        return out

    # ground points of rendered pixels (horizonator_pick_batch*: what is at this pixel)
    def pick(self, views, pixels):
        """views as render_batch takes them; pixels: (m, 2) (x, y) pairs asked of every view, or (n, m, 2) per view (x
        column, y row, 0 = top).  Returns an (n, m) structured array (GROUND_DTYPE): lat, lon, ele_m, distance_m of the
        ground point the pixel shows, range_m (bit-identical to the range image) and the triangle number; sky: triangle
        0xFFFFFFFF, range_m -1, the rest NaN (horizonator-batch.h).  Only the ground points leave the GPU."""
        n = len(views)
        px = np.asarray(pixels, dtype=np.int32)
        px = px.reshape(-1, 2) if px.ndim < 3 else px
        px = np.ascontiguousarray(np.broadcast_to(px, (n,) + px.shape[-2:]))
        m = px.shape[1]
        out = _pool.array((n, m), GROUND_DTYPE)
        _check(lib.horizonator_pick_batch, C.byref(self._ctx), n, self._views(views), m,
               px.ctypes.data if px.size else None, out.ctypes.data if out.size else None)
        return out

    def ground(self, views):
        """The ground point of every pixel: (lat, lon, ele, range), each (n, H, W) in image order (float64, float64,
        float32, float32; sky: NaN, NaN, NaN, -1).  n * H * W * 32 bytes cross the bus."""
        n = len(views)
        g = _pool.array((n, self.height, self.width), GROUND_DTYPE)
        _check(lib.horizonator_pick_batch, C.byref(self._ctx), n, self._views(views), 0, None,
               g.ctypes.data if g.size else None)
        return g["lat"], g["lon"], g["ele_m"], g["range_m"]

    def pick_device(self, views, d_pixels, d_ground, d_images=0, d_ranges=0, stream=0, m=None):
        """Device-memory variant.  d_pixels: an (n, m, 2) int32 CUDA tensor, an integer device address with `m` given,
        or None / 0 for every pixel; d_ground: a CUDA tensor or address of n * m (or n * H * W) ground_t, e.g. an
        (n, m, 32) uint8 tensor (.cpu().numpy().view(GROUND_DTYPE) reads it); d_images / d_ranges as render_batch_device
        (0 = not written); stream as render_batch_device."""
        if hasattr(d_pixels, "data_ptr"):
            if m is None:
                m = d_pixels.shape[-2]
            d_pixels = d_pixels.data_ptr()
        if hasattr(d_ground, "data_ptr"):
            d_ground = d_ground.data_ptr()
        d_images, d_ranges = (a.data_ptr() if hasattr(a, "data_ptr") else a for a in (d_images, d_ranges))
        _check(lib.horizonator_pick_batch_device, C.byref(self._ctx), len(views), self._views(views),
               int(m or 0), d_pixels or None, d_ground or None, d_images or None, d_ranges or None, stream or None)


class _PinnedBlock:
    def __init__(self, nbytes):
        self.ptr = lib.horizonator_host_alloc(nbytes)
        if not self.ptr:
            raise MemoryError("horizonator_host_alloc(%d) failed" % nbytes)

    def __del__(self):
        if getattr(self, "ptr", None) and lib is not None:
            lib.horizonator_host_free(self.ptr)
            self.ptr = None


class _PinnedLease:
    """Ties a pooled block to the lifetime of the numpy array built on it."""
    __slots__ = ("pool", "block", "nbytes")

    def __init__(self, pool, block, nbytes):
        self.pool, self.block, self.nbytes = pool, block, nbytes

    def __del__(self):
        pool = self.pool
        if pool is not None:
            pool._give_back(self.block, self.nbytes)


class _PinnedPool:
    """Recycles page-locked blocks for the arrays render() returns.  cudaMallocHost costs about a millisecond, so
    blocks are kept (up to `keep` bytes) and handed out again once the array that used them is gone."""

    def __init__(self, keep=1 << 30):
        self.free = {}          # nbytes -> [blocks]
        self.kept = 0
        self.keep = keep

    def array(self, shape, dtype):
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        n = max(count * dtype.itemsize, 1)
        blocks = self.free.get(n)
        if blocks:
            block = blocks.pop()
            self.kept -= n
        else:
            try:
                block = _PinnedBlock(n)
            except MemoryError:
                return np.empty(shape, dtype=dtype)      # out of page-locked memory: an ordinary array works too
        buf = (C.c_uint8 * n).from_address(block.ptr)
        buf._hz_lease = _PinnedLease(self, block, n)     # dies with the last view of buf
        return np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)

    def _give_back(self, block, n):
        if self.kept + n <= self.keep:
            self.free.setdefault(n, []).append(block)
            self.kept += n
        # else: the block is freed with its last reference (_PinnedBlock.__del__)


_pool = _PinnedPool()


def pinned_array(shape, dtype):
    """numpy array in page-locked host memory (horizonator_host_alloc); freed with the array."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    block = _PinnedBlock(max(n, 1))
    buf = (C.c_uint8 * max(n, 1)).from_address(block.ptr)
    buf._hz_block = block                 # keeps the allocation alive as long as any view of it
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
