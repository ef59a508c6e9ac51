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


def _declare(lib):
    P = C.POINTER
    ctx = P(context_t)
    f, d, i, b, vp, cp = C.c_float, C.c_double, C.c_int, C.c_bool, C.c_void_p, C.c_char_p
    sigs = {
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
    }
    for name, (res, args) in sigs.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise ImportError("%s is stale (no symbol %s): rebuild it with `python horizonator_b200/build.py`"
                              % (LIBRARY_PATH, name)) from None
        fn.restype = res
        fn.argtypes = args
    return lib


#: every symbol include/*.h declares (tests check that the library exports each of them)
EXPORTED_SYMBOLS = (
    "horizonator_init", "horizonator_deinit", "horizonator_resized", "horizonator_pan_zoom",
    "horizonator_move", "horizonator_set_zextents", "horizonator_redraw", "horizonator_pick",
    "horizonator_render_offscreen", "horizonator_x_from_az", "horizonator_project",
    "horizonator_unproject",
    "horizonator_dem_init", "horizonator_dem_deinit", "horizonator_dem_sample",
    "horizonator_dem_bounds_latlon_deg",
    "horizonator_render_batch_device", "horizonator_render_batch", "horizonator_render_wedge_device",
    "horizonator_download_mosaic", "horizonator_time_mosaic", "horizonator_last_render_stats",
    "horizonator_profile_enable", "horizonator_profile_read",
    "horizonator_host_alloc", "horizonator_host_free",
    "horizonator_render_counters", "horizonator_horizon_profile_device", "horizonator_set_earth_curvature", "horizonator_set_seam_wrap",
    "horizonator_peer_alloc", "horizonator_peer_open", "horizonator_peer_close", "horizonator_peer_free",
    "horizonator_render_wedge_peers", "horizonator_peer_barrier",
    "horizonator_render_wedge_host", "horizonator_host_register", "horizonator_host_unregister",
    "horizonator_debug_device_math", "horizonator_set_lod",
    "horizonator_viewshed_device", "horizonator_viewshed",
)

if not os.path.exists(LIBRARY_PATH):
    raise ImportError(
        "%s is missing: build it with `python horizonator_b200/build.py` (needs nvcc). "
        "horizonator_b200 has no CPU fallback." % LIBRARY_PATH)

lib = _declare(C.CDLL(LIBRARY_PATH))


def _enc(s):
    return None if s is None else os.fsencode(s)


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
        if not lib.horizonator_init(C.byref(self._ctx), lat, lon, None,
                                    int(width), int(height),
                                    int(render_radius_cells), float(render_radius_m),
                                    True, bool(render_texture), bool(SRTM1),
                                    _enc(dir_dems), _enc(dir_tiles), _enc(tiles_name), _enc(tiles_url_fmt),
                                    bool(allow_downloads)):
            raise RuntimeError("horizonator_init() failed")

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
        if not lib.horizonator_pan_zoom(C.byref(self._ctx), az_deg0, az_deg1):
            raise RuntimeError("horizonator_pan_zoom() failed")
        if lat > -1000.:
            if not lib.horizonator_move(C.byref(self._ctx), None, lat, lon):
                raise RuntimeError("horizonator_move() failed")
        if not lib.horizonator_set_zextents(C.byref(self._ctx), znear, zfar, znear_color, zfar_color):
            raise RuntimeError("horizonator_set_zextents() failed")
        # fresh arrays per call like the reference (pywrap.c:234-250), but out of a recycling pool of page-locked
        # blocks: the results then arrive by DMA instead of through the driver's pageable staging (3x faster for
        # 15 MB), and a block goes back to the pool when the caller drops the array
        image = _pool.array((H, W, 3), np.uint8) if return_image else None
        ranges = _pool.array((H, W), np.float32) if return_range else None
        if not lib.horizonator_render_offscreen(C.byref(self._ctx),
                                                image.ctypes.data if image is not None else None,
                                                ranges.ctypes.data if ranges is not None else None):
            raise RuntimeError("horizonator_render_offscreen() failed")
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
        if not lib.horizonator_set_zextents(C.byref(self._ctx), znear, zfar, znear_color, zfar_color):
            raise RuntimeError("horizonator_set_zextents() failed")

    def render_batch(self, views, return_image=True, return_range=True):
        """views: sequence of (lat, lon, az_deg0, az_deg1[, viewer_z]).  Host arrays (n,H,W,3), (n,H,W)."""
        n, W, H = len(views), self.width, self.height
        # page-locked blocks from the recycling pool, like render(): the copies of different views then run by DMA and
        # overlap the next views' kernels (into pageable arrays each copy would go through the driver's staging)
        image = _pool.array((n, H, W, 3), np.uint8) if return_image else None
        ranges = _pool.array((n, H, W), np.float32) if return_range else None
        if not lib.horizonator_render_batch(C.byref(self._ctx), n, self._views(views),
                                            image.ctypes.data if image is not None else None,
                                            ranges.ctypes.data if ranges is not None else None):
            raise RuntimeError("horizonator_render_batch() failed")
        return image, ranges

    def render_batch_device(self, views, d_images=0, d_ranges=0, stream=0):
        """Device-pointer variant: d_images / d_ranges are integer device addresses (e.g. tensor.data_ptr()),
        stream an integer cudaStream_t (0 = the context's own stream, synchronous)."""
        if not lib.horizonator_render_batch_device(C.byref(self._ctx), len(views), self._views(views),
                                                   d_images or None, d_ranges or None, stream or None):
            raise RuntimeError("horizonator_render_batch_device() failed")

    def render_wedge_device(self, x0, x1, d_image=0, d_ranges=0, stream=0):
        if not lib.horizonator_render_wedge_device(C.byref(self._ctx), int(x0), int(x1),
                                                   d_image or None, d_ranges or None, stream or None):
            raise RuntimeError("horizonator_render_wedge_device() failed")

    def render_wedge_host(self, x0, x1, image=None, ranges=None):
        """Columns [x0, x1) of the current view into FULL-size host arrays (H,W,3) uint8 / (H,W) float32."""
        if not lib.horizonator_render_wedge_host(C.byref(self._ctx), int(x0), int(x1),
                                                 image.ctypes.data if image is not None else None,
                                                 ranges.ctypes.data if ranges is not None else None):
            raise RuntimeError("horizonator_render_wedge_host() failed")

    def set_seam_wrap(self, on=True):
        """Opt-in (off by default; the reference drops them): draw triangles across the +-180 degree seam at both
        edges of a full-circle panorama.  See horizonator-batch.h."""
        if not lib.horizonator_set_seam_wrap(C.byref(self._ctx), bool(on)):
            raise RuntimeError("horizonator_set_seam_wrap() failed")

    def set_lod(self, max_cell_pixels=0.5):
        """Opt-in level of detail (0 = off, the default; the reference always draws every DEM cell): coarser far mesh
        where a coarser cell still is at most `max_cell_pixels` pixels across.  See horizonator-batch.h."""
        if not lib.horizonator_set_lod(C.byref(self._ctx), float(max_cell_pixels)):
            raise RuntimeError("horizonator_set_lod() failed")

    def set_earth_curvature(self, on=True, refraction=0.13):
        """Opt-in accuracy mode (off by default; the reference is flat-earth): see horizonator-batch.h."""
        if not lib.horizonator_set_earth_curvature(C.byref(self._ctx), bool(on), float(refraction)):
            raise RuntimeError("horizonator_set_earth_curvature() failed")

    # peer-memory assembly of wedge-sharded panoramas (horizonator-batch.h); used by sharding.PeerPanorama
    def peer_alloc(self, nbytes):
        """-> (device address, 64-byte handle) of a buffer other ranks can map."""
        ptr, handle = C.c_void_p(), (C.c_ubyte * 64)()
        if not lib.horizonator_peer_alloc(C.byref(self._ctx), nbytes, C.byref(ptr), C.byref(handle)):
            raise RuntimeError("horizonator_peer_alloc() failed")
        return ptr.value, bytes(handle)

    def peer_open(self, handle):
        ptr = C.c_void_p()
        if not lib.horizonator_peer_open(C.byref(self._ctx), (C.c_ubyte * 64).from_buffer_copy(handle), C.byref(ptr)):
            raise RuntimeError("horizonator_peer_open() failed")
        return ptr.value

    def peer_close(self, ptr):
        lib.horizonator_peer_close(C.byref(self._ctx), ptr)

    def peer_free(self, ptr):
        lib.horizonator_peer_free(C.byref(self._ctx), ptr)

    def peer_barrier(self, rank, d_flags, epoch, stream=0):
        """GPU-side barrier between ranks (horizonator_peer_barrier); d_flags: every rank's flag block address."""
        arr = (C.c_void_p * len(d_flags))(*d_flags)
        if not lib.horizonator_peer_barrier(C.byref(self._ctx), len(d_flags), int(rank), arr, int(epoch), stream or None):
            raise RuntimeError("horizonator_peer_barrier() failed")

    def render_wedge_peers(self, x0, x1, d_images, d_ranges, stream=0):
        """d_images / d_ranges: sequences of device addresses of every rank's full image / range buffer (or None)."""
        n = len(d_images) if d_images is not None else len(d_ranges)
        ai = (C.c_void_p * n)(*d_images) if d_images is not None else None
        ar = (C.c_void_p * n)(*d_ranges) if d_ranges is not None else None
        if not lib.horizonator_render_wedge_peers(C.byref(self._ctx), int(x0), int(x1), n, ai, ar, stream or None):
            raise RuntimeError("horizonator_render_wedge_peers() failed")

    def pan_zoom(self, az_deg0, az_deg1):
        if not lib.horizonator_pan_zoom(C.byref(self._ctx), az_deg0, az_deg1):
            raise RuntimeError("horizonator_pan_zoom() failed")

    def move(self, lat, lon, viewer_z=None):
        z = C.c_float(-1. if viewer_z is None else viewer_z)
        if not lib.horizonator_move(C.byref(self._ctx), C.byref(z), lat, lon):
            raise RuntimeError("horizonator_move() failed")
        return z.value

    def mosaic(self):
        """The decoded DEM square as the GPU holds it: (2R, 2R) int16, [j north][i east]."""
        n = 2 * self._ctx.dems.radius_cells
        out = np.empty((n, n), dtype=np.int16)
        if not lib.horizonator_download_mosaic(C.byref(self._ctx), out.ctypes.data):
            raise RuntimeError("horizonator_download_mosaic() failed")
        return out

    def time_mosaic(self, reps=10):
        ms = C.c_float(0)
        if not lib.horizonator_time_mosaic(C.byref(self._ctx), reps, C.byref(ms)):
            raise RuntimeError("horizonator_time_mosaic() failed")
        return ms.value

    def render_into(self, image, ranges):
        """horizonator_render_offscreen() with the current state into caller-owned arrays (either may be
        None): no allocation, and DMA speed when the arrays come from pinned_array()."""
        if not lib.horizonator_render_offscreen(C.byref(self._ctx),
                                                image.ctypes.data if image is not None else None,
                                                ranges.ctypes.data if ranges is not None else None):
            raise RuntimeError("horizonator_render_offscreen() failed")

    def profile(self, on=True):
        """Record CUDA events around every kernel of every render from now on (see profile_read)."""
        if not lib.horizonator_profile_enable(C.byref(self._ctx), bool(on)):
            raise RuntimeError("horizonator_profile_enable() failed")

    def profile_read(self):
        """Mean device ms per render of each kernel since the last read, and the number of renders."""
        ms = (C.c_float * 6)()
        n = C.c_int(0)
        if not lib.horizonator_profile_read(C.byref(self._ctx), C.byref(ms), C.byref(n)):
            raise RuntimeError("horizonator_profile_read() failed")
        return {"prepare": ms[0], "near": ms[1], "big_near": ms[2], "march": ms[3], "big_far": ms[4],
                "resolve": ms[5], "renders": n.value}

    def last_render_stats(self):
        out = (C.c_uint * 5)()
        if not lib.horizonator_last_render_stats(C.byref(self._ctx), C.byref(out)):
            raise RuntimeError("horizonator_last_render_stats() failed")
        return {"big_entries": out[0], "big_capacity": out[1], "launches": out[2], "device": out[3],
                "triangles_rasterised": out[4]}

    COUNTER_NAMES = ("tiles", "tiles_far", "tiles_window", "tiles_occluded",
                     "blocks", "blocks_far", "blocks_window", "blocks_occluded",
                     "blocks_meshed", "triangles", "big_entries")

    def render_counters(self):
        """Culling counters of the most recent render (horizonator_render_counters)."""
        out = (C.c_uint * 16)()
        if not lib.horizonator_render_counters(C.byref(self._ctx), C.byref(out)):
            raise RuntimeError("horizonator_render_counters() failed")
        return dict(zip(self.COUNTER_NAMES, out))

    def horizon_profile_device(self, d_ranges, n, d_rows, d_range, stream=0):
        """Per-column topmost terrain (row, range) of n device range images; all arguments device addresses."""
        if not lib.horizonator_horizon_profile_device(C.byref(self._ctx), d_ranges, int(n), d_rows, d_range,
                                                      stream or None):
            raise RuntimeError("horizonator_horizon_profile_device() failed")

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
        if not lib.horizonator_viewshed(C.byref(self._ctx), n, self._eyes(views), float(target_height),
                                        words.ctypes.data, cnt.ctypes.data if counts else None):
            raise RuntimeError("horizonator_viewshed() failed")
        bits = np.unpackbits(words.view(np.uint8), axis=-1, bitorder="little")[..., :N].astype(bool)
        return (bits, cnt) if counts else bits

    def viewshed_device(self, views, d_masks=0, d_counts=0, target_height=0., stream=0):
        """Device-pointer variant: d_masks (n, N, (N+31)//32) uint32 words, overwritten; d_counts (N, N) uint32,
        added to.  Integer device addresses, either may be 0 (not both); stream as render_batch_device."""
        if not lib.horizonator_viewshed_device(C.byref(self._ctx), len(views), self._eyes(views), float(target_height),
                                               d_masks or None, d_counts or None, stream or None):
            raise RuntimeError("horizonator_viewshed_device() failed")


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
