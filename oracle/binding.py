"""oracle/binding.py -- TEST INFRASTRUCTURE.  ctypes access to the CPU oracle.

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this.

  Oracle      liboracle.so: the CPU restatement (horizonator_oracle.c + gl_pipeline.c)
  Reference   _ref/libhorizonator_ref.so: the reference's own horizonator-lib.c + dem.c, compiled
              unmodified from /root/reference on the fake GL of oracle/fakegl (prebuilt .so travels)
  MesaReference  _ref/libhorizonator_mesa.so: the same two files, unmodified, on a REAL OpenGL driver -- the
              Mesa llvmpipe libGL inside the image (oracle/mesa/): what pins the GL rules of gl_pipeline.c
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "liboracle.so")
REF_SO = os.path.join(HERE, "_ref", "libhorizonator_ref.so")
MESA_SO = os.path.join(HERE, "_ref", "libhorizonator_mesa.so")


class _dem_context_t(C.Structure):
    """/root/reference/dem.h: horizonator_dem_context_t (352 bytes).  Declared here, not imported from the product
    package, so that nothing of the product is loaded by the reference arm."""
    _fields_ = [("dems", (C.c_void_p * 4) * 4), ("mmap_sizes", (C.c_size_t * 4) * 4), ("mmap_fd", (C.c_int * 4) * 4),
                ("origin_dem_lon_lat", C.c_int * 2), ("origin_dem_cellij", C.c_int * 2), ("Ndems_ij", C.c_int * 2),
                ("radius_cells", C.c_int), ("cells_per_deg", C.c_int)]


class _offscreen_t(C.Structure):
    _fields_ = [("inited", C.c_bool), ("frameBufID", C.c_uint32), ("renderBufID", C.c_uint32), ("depthBufID", C.c_uint32),
                ("width", C.c_int), ("height", C.c_int)]


class context_t(C.Structure):
    """/root/reference/horizonator.h: horizonator_context_t (472 bytes)."""
    _fields_ = [("Ntriangles", C.c_int), ("render_texture", C.c_bool), ("use_glut", C.c_bool), ("glut_window", C.c_int),
                ("uniforms", C.c_int32 * 17), ("program", C.c_uint32), ("viewer_lat", C.c_float), ("viewer_lon", C.c_float),
                ("dems", _dem_context_t), ("offscreen", _offscreen_t)]


assert C.sizeof(_dem_context_t) == 352 and C.sizeof(context_t) == 472


def build(ref=True):
    """make liboracle.so (+ _ref, on the fake GL and on Mesa, when /root/reference is present)."""
    targets = ["liboracle.so"] + (["ref", "mesa"] if ref else [])
    subprocess.run(["make", "-s", "-C", HERE] + targets, check=True)


def have_ref():
    return os.path.exists(REF_SO)


def mesa_libgl():
    """Path of the Mesa libGL the llvmpipe build links to (inside Nsight Compute), or None."""
    import glob
    hits = sorted(glob.glob("/opt/nvidia/nsight-compute/*/host/linux-desktop-glibc_2_11_3-x64/Mesa/libGL.so.1"))
    return hits[0] if hits else None


def have_mesa():
    """True where the reference-on-llvmpipe build exists AND the libGL it was linked to is in the image."""
    if not os.path.exists(MESA_SO):
        return False
    out = subprocess.run(["ldd", MESA_SO], capture_output=True, text=True).stdout
    return "not found" not in out and "libGL.so.1" in out


class Oracle:
    """CPU restatement; same call sequence as the reference's Python type."""
    _lib = None

    @classmethod
    def lib(cls):
        if cls._lib is None:
            if not os.path.exists(ORACLE_SO):
                build(ref=False)
            L = C.CDLL(ORACLE_SO)
            f, i, b, vp = C.c_float, C.c_int, C.c_bool, C.c_void_p
            L.oracle_init.restype = vp
            L.oracle_init.argtypes = [f, f, C.POINTER(f), i, i, i, f, b, C.c_char_p]
            L.oracle_deinit.argtypes = [vp]
            L.oracle_move.restype = b
            L.oracle_move.argtypes = [vp, C.POINTER(f), f, f]
            L.oracle_pan_zoom.restype = b
            L.oracle_pan_zoom.argtypes = [vp, f, f]
            L.oracle_set_zextents.restype = b
            L.oracle_set_zextents.argtypes = [vp, f, f, f, f]
            L.oracle_render_offscreen.restype = b
            L.oracle_render_offscreen.argtypes = [vp, vp, vp]
            L.oracle_dem_sample.restype = C.c_int16
            L.oracle_dem_sample.argtypes = [vp, i, i]
            L.oracle_get_dem_geometry.argtypes = [vp, C.POINTER(C.c_int * 8)]
            L.oracle_get_viewer.argtypes = [vp, C.POINTER(C.c_float * 4)]
            L.oracle_set_threads.argtypes = [vp, i]
            L.oracle_set_curvature.argtypes = [vp, f]
            L.oracle_set_seam_wrap.argtypes = [vp, b]
            L.oracle_vertex_stage.restype = f
            L.oracle_vertex_stage.argtypes = [vp, vp]
            L.oracle_read_keys.restype = b
            L.oracle_read_keys.argtypes = [vp, i, i, f, f, f, f, vp, vp]
            L.glp_draw_keys.restype = i
            L.glp_draw_keys.argtypes = [vp, i, i, vp, i, f, vp, i]
            cls._lib = L
        return cls._lib

    def __init__(self, lat, lon, width, height, SRTM1=False, dir_dems=None,
                 render_radius_cells=-1, render_radius_m=-1., viewer_z=None, threads=1):
        L = self.lib()
        z = C.c_float(-1. if viewer_z is None else viewer_z)
        self.h = L.oracle_init(lat, lon, C.byref(z), width, height, render_radius_cells, render_radius_m,
                               SRTM1, os.fsencode(dir_dems))
        if not self.h:
            raise RuntimeError("oracle_init() failed")
        self.viewer_z = z.value
        self.W, self.H = width, height
        L.oracle_set_threads(self.h, threads)

    def close(self):
        if self.h:
            self.lib().oracle_deinit(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def move(self, lat, lon, viewer_z=None):
        z = C.c_float(-1. if viewer_z is None else viewer_z)
        assert self.lib().oracle_move(self.h, C.byref(z), lat, lon)
        return z.value

    def set_seam_wrap(self, on=True):
        """Opt-in extension (not in the reference): seam-straddling triangles drawn at both edges."""
        self.lib().oracle_set_seam_wrap(self.h, on)

    def set_curvature(self, coefficient):
        """Opt-in extension (not in the reference): height drop = coefficient * distance^2; 0 = off."""
        self.lib().oracle_set_curvature(self.h, coefficient)

    def dem_geometry(self):
        out = (C.c_int * 8)()
        self.lib().oracle_get_dem_geometry(self.h, C.byref(out))
        return dict(origin_dem_lon_lat=(out[0], out[1]), origin_dem_cellij=(out[2], out[3]),
                    Ndems_ij=(out[4], out[5]), radius_cells=out[6], cells_per_deg=out[7])

    def viewer(self):
        out = (C.c_float * 4)()
        self.lib().oracle_get_viewer(self.h, C.byref(out))
        return dict(viewer_cell_i=out[0], viewer_cell_j=out[1], viewer_z=out[2], cos_viewer_lat=out[3])

    def dem_sample(self, i, j):
        return self.lib().oracle_dem_sample(self.h, i, j)

    def mosaic(self):
        n = 2 * self.dem_geometry()["radius_cells"]
        L = self.lib()
        return np.array([[L.oracle_dem_sample(self.h, i, j) for i in range(n)] for j in range(n)], dtype=np.int16)

    def _set_view(self, az_deg0, az_deg1, lat, lon, znear, zfar, znear_color, zfar_color):
        L = self.lib()
        if znear_color < 0:
            znear_color = znear
        if zfar_color < 0:
            zfar_color = zfar
        assert L.oracle_pan_zoom(self.h, az_deg0, az_deg1)
        if lat > -1000.:
            self.move(lat, lon)
        if not L.oracle_set_zextents(self.h, znear, zfar, znear_color, zfar_color):
            raise RuntimeError("oracle_set_zextents() failed")

    def vertex_stage(self, az_deg0, az_deg1, lat=-1000., lon=-1000., znear=100., zfar=40000.,
                     znear_color=-1., zfar_color=-1.):
        """This oracle's vertex stage for the view render() would draw: (glp_vtx_t records [j * N + i], seam period)"""
        self._set_view(az_deg0, az_deg1, lat, lon, znear, zfar, znear_color, zfar_color)
        n = 2 * self.dem_geometry()["radius_cells"]
        from oracle.vertex import VTX
        vtx = np.empty(n * n, VTX)
        period = self.lib().oracle_vertex_stage(self.h, vtx.ctypes.data)
        return vtx, period

    def render(self, az_deg0, az_deg1, lat=-1000., lon=-1000., znear=100., zfar=40000.,
               znear_color=-1., zfar_color=-1.):
        L = self.lib()
        self._set_view(az_deg0, az_deg1, lat, lon, znear, zfar, znear_color, zfar_color)
        image = np.empty((self.H, self.W, 3), np.uint8)
        ranges = np.empty((self.H, self.W), np.float32)
        assert L.oracle_render_offscreen(self.h, image.ctypes.data, ranges.ctypes.data)
        return image, ranges


KEY_Q_SHIFT, KEY_ID_MASK, Z24_MAX = 37, 0x1FFFFFFF, 0xFFFFFF     # oracle/gl_pipeline.h


def draw_keys(vtx, N, W, H, seam_period=0.0, levels=None, threads=None):
    """glp_draw_keys(): the visibility key of every pixel ((H, W) uint64, GL row order, bottom row first) of every
    triangle of the N x N vertices vtx (oracle.vertex.VTX records [j * N + i]), unculled; levels: int8 [tj][ti] level
    of detail per tile (oracle.vertex.tile_levels), None = the reference's mesh"""
    from oracle.vertex import VTX, n_tiles
    vtx = np.ascontiguousarray(vtx, VTX)
    assert vtx.shape == (N * N,)
    if levels is not None:
        levels = np.ascontiguousarray(levels, np.int8)
        assert levels.shape == (n_tiles(N), n_tiles(N))
    keys = np.empty((H, W), np.uint64)
    assert Oracle.lib().glp_draw_keys(keys.ctypes.data, W, H, vtx.ctypes.data, N, seam_period,
                                      None if levels is None else levels.ctypes.data, threads or os.cpu_count() or 1)
    return keys


def read_keys(keys, az_deg0, az_deg1, znear, zfar):
    """image (H, W, 3) and ranges (H, W) of keys, top row first, by oracle_render_offscreen()'s read-back"""
    H, W = keys.shape
    keys = np.ascontiguousarray(keys, np.uint64)
    image = np.empty((H, W, 3), np.uint8)
    ranges = np.empty((H, W), np.float32)
    assert Oracle.lib().oracle_read_keys(keys.ctypes.data, W, H, az_deg0, az_deg1, znear, zfar, image.ctypes.data,
                                         ranges.ctypes.data)
    return image, ranges


def key_triangles(keys, N, levels=None):
    """(H, W) uint32, top row first: the triangle number each key holds, with the level of detail of its cell's tile
    in bits [30:29] as horizonator_pick_batch() reports it; 0xFFFFFFFF where nothing was drawn"""
    from oracle.vertex import LOD_SHIFT, TILE_CELLS
    keys = keys[::-1]
    sky = (keys >> np.uint64(KEY_Q_SHIFT)) >= Z24_MAX
    tri = ((keys >> np.uint64(8)) & np.uint64(KEY_ID_MASK)).astype(np.uint32)
    if levels is not None:
        cell = tri >> 1
        tj, ti = (cell // (N - 1)) // TILE_CELLS, (cell % (N - 1)) // TILE_CELLS
        tri |= levels[np.where(sky, 0, tj), np.where(sky, 0, ti)].astype(np.uint32) << LOD_SHIFT
    return np.where(sky, np.uint32(0xFFFFFFFF), tri)


class Reference:
    """The reference's horizonator-lib.c + dem.c (unmodified) on the fake GL.  One live instance at a time:
    the fake GL, like the code it serves, keeps one current program/framebuffer."""
    _lib = None
    SO = REF_SO
    FAKE_GL = True

    @classmethod
    def lib(cls):
        if cls.__dict__.get("_lib") is None:
            L = C.CDLL(cls.SO)
            f, d, i, b, vp, cp = C.c_float, C.c_double, C.c_int, C.c_bool, C.c_void_p, C.c_char_p
            L.horizonator_init.restype = b
            L.horizonator_init.argtypes = [vp, f, f, C.POINTER(f), i, i, i, f, b, b, b, cp, cp, cp, cp, b]
            L.horizonator_move.restype = b
            L.horizonator_move.argtypes = [vp, C.POINTER(f), f, f]
            L.horizonator_pan_zoom.restype = b
            L.horizonator_pan_zoom.argtypes = [vp, f, f]
            L.horizonator_set_zextents.restype = b
            L.horizonator_set_zextents.argtypes = [vp, f, f, f, f]
            L.horizonator_render_offscreen.restype = b
            L.horizonator_render_offscreen.argtypes = [vp, vp, vp]
            L.horizonator_pick.restype = b
            L.horizonator_pick.argtypes = [vp, C.POINTER(f), C.POINTER(f), i, i]
            L.horizonator_dem_sample.restype = C.c_int16
            L.horizonator_dem_sample.argtypes = [vp, i, i]
            L.horizonator_dem_init.restype = b
            L.horizonator_dem_init.argtypes = [vp, f, f, i, f, cp, b]
            L.horizonator_dem_deinit.argtypes = [vp]
            L.horizonator_x_from_az.restype = b
            L.horizonator_x_from_az.argtypes = [C.POINTER(d), C.POINTER(d), d, d, d, i]
            L.horizonator_project.restype = b
            L.horizonator_project.argtypes = [C.POINTER(d)] * 3 + [d] * 9 + [i, i]
            L.horizonator_unproject.restype = b
            L.horizonator_unproject.argtypes = [C.POINTER(f), C.POINTER(f), i, i] + [d] * 7 + [i, i]
            L.horizonator_deinit.restype = None
            L.horizonator_deinit.argtypes = [vp]
            if cls.FAKE_GL:
                L.fakegl_set_threads.argtypes = [i]
            else:
                L.glut_glx_renderer.restype = cp
                L.glut_glx_version.restype = cp
            cls._lib = L
        return cls._lib

    def __init__(self, lat, lon, width, height, SRTM1=False, dir_dems=None,
                 render_radius_cells=-1, render_radius_m=-1., viewer_z=None, threads=1):
        L = self.lib()
        self._set_threads(threads)
        self.ctx = None
        ctx = context_t()
        z = C.c_float(-1. if viewer_z is None else viewer_z)
        if not L.horizonator_init(C.byref(ctx), lat, lon, C.byref(z), width, height,
                                  render_radius_cells, render_radius_m, True, False, SRTM1,
                                  os.fsencode(dir_dems), None, None, None, False):
            raise RuntimeError("reference horizonator_init() failed")
        self.ctx = ctx
        self.viewer_z = z.value
        self.W, self.H = width, height

    def _set_threads(self, threads):
        self.lib().fakegl_set_threads(threads)

    def close(self):
        """horizonator_deinit() (horizonator-lib.c:682-689): gives the GL context back."""
        if self.ctx is not None:
            self.lib().horizonator_deinit(C.byref(self.ctx))
            self.lib().horizonator_dem_deinit(C.byref(self.ctx.dems))
            self.ctx = None

    def move(self, lat, lon, viewer_z=None):
        z = C.c_float(-1. if viewer_z is None else viewer_z)
        assert self.lib().horizonator_move(C.byref(self.ctx), C.byref(z), lat, lon)
        return z.value

    def dem_sample(self, i, j):
        return self.lib().horizonator_dem_sample(C.byref(self.ctx.dems), i, j)

    def mosaic(self):
        """The whole DEM square through the reference's own horizonator_dem_sample() (dem.c:264-309), one call per
        cell as horizonator-lib.c:435-439 does it, in a C loop (oracle/fakegl/fakegl.c: ref_sample_square)."""
        n = 2 * self.ctx.dems.radius_cells
        out = np.empty((n, n), np.int16)
        L = self.lib()
        L.ref_sample_square.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.ref_sample_square(C.byref(self.ctx.dems), n, out.ctypes.data)
        return out

    def render(self, az_deg0, az_deg1, lat=-1000., lon=-1000., znear=100., zfar=40000.,
               znear_color=-1., zfar_color=-1.):
        L = self.lib()
        if znear_color < 0:
            znear_color = znear
        if zfar_color < 0:
            zfar_color = zfar
        assert L.horizonator_pan_zoom(C.byref(self.ctx), az_deg0, az_deg1)
        if lat > -1000.:
            self.move(lat, lon)
        if not L.horizonator_set_zextents(C.byref(self.ctx), znear, zfar, znear_color, zfar_color):
            raise RuntimeError("reference horizonator_set_zextents() failed")
        image = np.empty((self.H, self.W, 3), np.uint8)
        ranges = np.empty((self.H, self.W), np.float32)
        assert L.horizonator_render_offscreen(C.byref(self.ctx), image.ctypes.data, ranges.ctypes.data)
        return image, ranges


class ReferenceDem:
    """Only the DEM layer of the reference (dem.c, unmodified, out of _ref/libhorizonator_ref.so): horizonator_dem_init()
    and the whole square through horizonator_dem_sample().  No GL context, no mesh."""

    def __init__(self, lat, lon, SRTM1=False, dir_dems=None, render_radius_cells=-1, render_radius_m=-1., threads=1):
        self.L = Reference.lib()
        self.L.fakegl_set_threads(threads)
        self.dems = _dem_context_t()
        if not self.L.horizonator_dem_init(C.byref(self.dems), lat, lon, render_radius_cells, render_radius_m,
                                           os.fsencode(dir_dems), SRTM1):
            self.dems = None
            raise RuntimeError("reference horizonator_dem_init() failed")

    def mosaic(self):
        n = 2 * self.dems.radius_cells
        out = np.empty((n, n), np.int16)
        self.L.ref_sample_square.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        self.L.ref_sample_square(C.byref(self.dems), n, out.ctypes.data)
        return out

    def close(self):
        if self.dems is not None:
            self.L.horizonator_dem_deinit(C.byref(self.dems))
            self.dems = None

    def __del__(self):
        self.close()


class MesaReference(Reference):
    """The reference's horizonator-lib.c + dem.c (unmodified) on Mesa's llvmpipe: a real OpenGL implementation
    (shader compiler, clipper, rasteriser, depth buffer, read-back), not a restatement.  One live instance per
    process at a time (one GLX context); close() before making the next.  llvmpipe sizes its rasteriser thread
    pool when the first context is created (LP_NUM_THREADS, default: all cores, at most 16); its vertex and
    geometry stages run on the calling thread."""
    _lib = None
    SO = MESA_SO
    FAKE_GL = False

    def _set_threads(self, threads):
        if threads and threads > 0:
            os.environ.setdefault("LP_NUM_THREADS", str(min(int(threads), 16)))

    def gl_strings(self):
        L = self.lib()
        return L.glut_glx_version().decode(), L.glut_glx_renderer().decode()
