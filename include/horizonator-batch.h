/* horizonator-batch.h -- additive entry points of the B200-native libhorizonator.
 *
 * The reference (dkogan/horizonator) has no counterpart for these: its only render call is
 * horizonator_render_offscreen() (horizonator.h:165-169), one view at a time into host
 * memory.  horizonator.h keeps that ABI untouched; everything new lives here.
 *
 * Same conventions: plain C, plain pointers and sizes, `bool` returns with a MSG() line on
 * stderr on failure.  "Device pointer" means memory of the CUDA device the context was
 * created on (e.g. torch tensor .data_ptr()); `stream` is a cudaStream_t passed as void*
 * (NULL = the context's own stream; the call then waits for completion before returning,
 * otherwise it only enqueues work and the caller synchronises).
 */
#pragma once

#include <stddef.h>

#include "horizonator.h"

#ifdef __cplusplus
extern "C" {
#endif

/* one view of a batch: an eye position inside the loaded DEM square and an azimuth window */
typedef struct
{
    float lat, lon;
    float viewer_z;          /* < 0: highest of the 4 surrounding samples + 1 m (as horizonator_move) */
    float az_deg0, az_deg1;  /* as horizonator_pan_zoom */
} horizonator_view_t;

/* Renders n views with the context's current z extents and image size (W x H).
 * d_images: n*H*W*3 bytes (B,G,R, top row first) or NULL; d_ranges: n*H*W floats or NULL;
 * both DEVICE pointers.  Leaves the context's own eye/azimuth state as it was.
 * The views are rendered in chunks that share every kernel launch (8 to 64 views each, spread over up to 4 streams):
 * throughput grows with n up to about 256 views per call (measured at 3600x600: 16 views 16 k panoramas/s, 64 views
 * 26 k, 256 views 33 k); each view in flight takes ~140 MB of scratch, allocated on first use. */
bool horizonator_render_batch_device(const horizonator_context_t* ctx,
                                     int n, const horizonator_view_t* views,
                                     void* d_images, void* d_ranges,
                                     void* stream);

/* Same, into HOST memory (images/ranges as in horizonator_render_offscreen, n of each). */
bool horizonator_render_batch(const horizonator_context_t* ctx,
                              int n, const horizonator_view_t* views,
                              char* images, float* ranges);

/* Renders only columns [x0, x1) of the context's current W x H panorama (current eye, azimuth
 * window and z extents) into DEVICE slabs d_image: H*(x1-x0)*3 bytes, d_ranges: H*(x1-x0)
 * floats (either may be NULL).  The columns are bit-identical to the same columns of a full
 * render: the projection, the quarter-width triangle discard (geometry.glsl:21-27) and the
 * depth test all use the full window; only the set of pixels written differs.  This is the
 * unit of work for splitting one giant panorama across GPUs by azimuth wedge. */
bool horizonator_render_wedge_device(const horizonator_context_t* ctx,
                                     int x0, int x1,
                                     void* d_image, void* d_ranges,
                                     void* stream);

/* The same columns into HOST memory laid out as the FULL panorama: image = H*W*3 bytes, ranges = H*W floats (as
 * horizonator_render_offscreen() takes them; either may be NULL), of which only columns [x0, x1) are written.
 * Synchronous.  Several contexts -- one per GPU, in one process or in several that share the buffer -- can fill
 * one panorama this way, each over its own PCIe link; page-lock the buffer (horizonator_host_alloc(), or
 * horizonator_host_register() for memory that exists already, e.g. a shared mapping) for DMA speed. */
bool horizonator_render_wedge_host(const horizonator_context_t* ctx,
                                   int x0, int x1,
                                   char* image, float* ranges);
bool horizonator_host_register(void* p, size_t bytes);
bool horizonator_host_unregister(void* p);

/* A wedge-sharded panorama assembled by the renderer itself over NVLink: instead of rendering its wedge
 * into a private slab that a collective then gathers, a rank's final kernel stores the wedge's pixels
 * straight into the FULL W x H image / range buffers of every rank (peer memory).
 *   horizonator_peer_alloc()   allocates such a full-size buffer on this context's device and returns a
 *                              64-byte inter-process handle for it (cudaIpcMemHandle_t)
 *   horizonator_peer_open()    maps another rank's buffer from its handle (ranks are separate processes;
 *                              how the handles travel is the caller's business -- the Python driver
 *                              uses torch.distributed.all_gather_object)
 *   horizonator_render_wedge_peers()  renders columns [x0,x1) of the context's current view and writes
 *                              them into column x0.. of each of the n_peers (1..8) destinations;
 *                              d_images / d_ranges are arrays of n_peers device pointers (either array may
 *                              be NULL).  The destinations are complete once EVERY rank's call has finished
 *                              on its stream: synchronise the ranks (a barrier) before reading them.
 *   horizonator_peer_close() / horizonator_peer_free()  undo open / alloc. */
bool horizonator_peer_alloc(const horizonator_context_t* ctx, size_t bytes, void** d_ptr, unsigned char handle[64]);
bool horizonator_peer_open(const horizonator_context_t* ctx, const unsigned char handle[64], void** d_ptr);
bool horizonator_peer_close(const horizonator_context_t* ctx, void* d_ptr);
bool horizonator_peer_free(const horizonator_context_t* ctx, void* d_ptr);
bool horizonator_render_wedge_peers(const horizonator_context_t* ctx, int x0, int x1, int n_peers,
                                    void* const* d_images, void* const* d_ranges, void* stream);

/* Barrier between the ranks of such a panorama ON THE GPUS (no host synchronisation, no collective
 * library): d_flags[r] is rank r's flag block -- HORIZONATOR_PEER_FLAG_BYTES bytes from
 * horizonator_peer_alloc(), zeroed once, mapped by every rank -- and `epoch` a number that every rank
 * increases by one per barrier.  Enqueued on `stream`: work queued after it starts once every rank's
 * stream has reached its own barrier of the same epoch, and sees everything those streams wrote before.
 * A rank that does not arrive within a few tenths of a second is given up on: the barrier returns and the
 * word at index 8 of the caller's own flag block counts the time-outs. */
#define HORIZONATOR_PEER_FLAG_BYTES 64
bool horizonator_peer_barrier(const horizonator_context_t* ctx, int n_ranks, int rank, void* const* d_flags,
                              unsigned int epoch, void* stream);

/* Opt-in accuracy mode; OFF by default, and off in every parity test: the reference renders a flat
 * tangent plane and says so (vertex.glsl:65-88: "31 m vertical error at 20 km", README.org:158-161).
 * When on, a point at horizontal distance d appears lower by (1 - refraction) * d^2 / (2 * 6371000 m)
 * -- the earth's curvature reduced by standard atmospheric refraction (refraction ~ 0.13; 0 = pure
 * geometry) -- in the elevation angle and in the slant range of every vertex.  Applies to all
 * later renders of the context. */
bool horizonator_set_earth_curvature(const horizonator_context_t* ctx, bool on, float refraction);

/* Opt-in, OFF by default and in every parity test: the reference DROPS every triangle whose vertices lie
 * on both sides of the window's +-180-degree seam (geometry.glsl:15-27 discards anything wider than a
 * quarter of the window), which leaves a gap up to one DEM cell wide at the left and right edge of a
 * full-circle panorama.  When on, such a triangle is drawn twice instead, once at each edge (its
 * vertices moved by one period of the azimuth mapping), so a 360-degree panorama closes.  Triangles
 * that are too wide for another reason stay dropped. */
bool horizonator_set_seam_wrap(const horizonator_context_t* ctx, bool on);

/* Opt-in level of detail; OFF (0) by default and in every parity test: the reference draws every cell of the DEM
 * however far away it is (README.org:169-185 lists a coarser far mesh as future work).  With max_cell_pixels > 0 the
 * parts of the mesh beyond the foreground are drawn with every 2nd or 4th vertex only -- cells of 2x2 or 4x4 DEM cells
 * -- wherever such a coarser cell, seen from the nearest edge of its distance band, is still at most max_cell_pixels
 * pixels across (0.5 is a sensible value: half a pixel).  The foreground is never coarsened.  Where two levels meet,
 * hairline cracks are possible; the image differs from the full render only by sub-pixel shifts of far silhouettes
 * (tests/test_gpu_large.py reports the differences), and views that see much distant terrain render several times
 * faster.  Applies to all later renders of the context. */
bool horizonator_set_lod(const horizonator_context_t* ctx, float max_cell_pixels);

/* Test hook: the renderer's own fp32 angle functions (csrc/hz_math.cuh) evaluated on the current CUDA device for n
 * argument sets in host arrays: az[k] = atan2(e[k], north[k]) (vertex.glsl:136), el[k] = atan(h[k] / sqrt(d2[k]))
 * (vertex.glsl:153).  tests/test_device_math.py measures their error in ulp against double precision. */
bool horizonator_debug_device_math(int n, const float* e, const float* north, const float* h, const float* d2,
                                   float* az, float* el);

/* Page-locked host memory for output buffers.  horizonator_render_offscreen() and
 * horizonator_render_batch() accept any host pointer; into memory from this allocator (or any
 * other CUDA-registered host memory) the results arrive by DMA at PCIe speed, into ordinary
 * pageable memory through the driver's staging copy (about 3x slower for a 15 MB result). */
void* horizonator_host_alloc(size_t bytes);
void  horizonator_host_free(void* p);

/* Copies the decoded DEM square (2R x 2R int16, row j = north index, column i = east index,
 * tightly packed) from the device to host memory.  For tests of the decode/stitch kernel. */
bool horizonator_download_mosaic(const horizonator_context_t* ctx, int16_t* mosaic);

/* Re-runs the decode/stitch kernel `reps` times and reports the mean device time per run in
 * milliseconds (CUDA events on the context's stream).  For benchmarks of the init path. */
bool horizonator_time_mosaic(const horizonator_context_t* ctx, int reps, float* ms_per_run);

/* Per-column horizon of n range images (device memory, n*H*W floats as the render calls
 * write them): d_rows[n*W] = row (0 = top) of the topmost terrain pixel of each column or -1,
 * d_range[n*W] = the range there or -1.  The reduced product of a viewpoint batch: a few
 * bytes per column instead of a full image. */
bool horizonator_horizon_profile_device(const horizonator_context_t* ctx,
                                        const void* d_ranges, int n,
                                        void* d_rows, void* d_range,
                                        void* stream);

/* Viewsheds: which vertices of the loaded DEM square each of n views sees, and for every vertex from how many of them.
 *
 * Definition (R2, the ray-casting viewshed of Franklin & Ray; the GPU kernel and the test oracle agree bit for bit):
 *   - Domain: the N x N vertices (i, j) of the loaded square (N = 2R), indexed like horizonator_download_mosaic()
 *     (row j north, column i east).  The point tested is the vertex's terrain height plus target_height_m.
 *   - Eye: as horizonator_move() computes it from lat, lon and viewer_z (< 0: the highest of the 4 surrounding
 *     samples + 1 m), in float.  az_deg0 / az_deg1 are ignored: a viewshed covers the full circle.  The eye's cell
 *     coordinates must lie in [0, N-1); otherwise the call fails (the render calls accept such eyes).
 *   - Metres: east and north offsets by the renderer's axis-table formulas (vertex.glsl:128-130) evaluated at the
 *     (possibly fractional) cell coordinate; the apparent height of a point at horizontal distance^2 d2 with terrain
 *     height z is z - viewer_z - curvature * d2, so horizonator_set_earth_curvature() applies (off by default).
 *   - Rays: one per boundary vertex of the square, 4N - 4.  A ray with |di| >= |dj| (di, dj: target minus eye, in
 *     cells) steps over the integer columns i strictly beyond the eye up to the target's; at column i,
 *     y = eye_j + (i - eye_i) * (dj / di), the surface is the linear interpolation between rows floor(y) and
 *     floor(y) + 1 of column i (a grid edge, hence exact on the mesh's triangles; the rows clamped to [0, N-2] and
 *     [1, N-1]), and its horizon slope is s = apparent height / horizontal distance.  The vertex that step decides is
 *     (i, rint(y)) (clamped to [0, N-1]): visible iff (its apparent height + target_height_m) / its own horizontal
 *     distance >= the largest s of the ray's EARLIER steps (-inf at the first step).  Rays with |dj| > |di| step
 *     over rows the same way, axes swapped.
 *   - A vertex is visible iff some ray finds it visible; the four vertices around the eye are visible.
 *   - fp32, every operation rounded once in the order written in hz_kernels.cu (k_viewshed) and
 *     oracle/viewshed_oracle.c (vs_oracle_r2).
 * R2 is an approximation of line of sight: on seeded synthetic terrain it disagrees with the exact line of sight on
 * the same triangulation on about 1 % of the vertices (DESIGN.md, viewsheds).
 *
 * masks: n x N x W32 uint32 (W32 = (N + 31) / 32; cell i of row j = bit (i & 31) of word [j][i >> 5], unused bits
 *        0), overwritten;
 * counts: N x N uint32, += the number of the n views that see each cell (the caller zeroes it; several calls and
 *        several ranks can add into one buffer);
 * either may be NULL, not both.  n = 0 does nothing.  Both DEVICE pointers here, stream as for the batch render.
 * Sizes at N = 11716 (150 km of SRTM1): one mask 17.2 MB, the counts 549 MB.  A call that wants only counts uses a
 * scratch of up to 64 masks, allocated on first use; the views go in chunks of up to 64 per kernel launch. */
bool horizonator_viewshed_device(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                                 float target_height_m, void* d_masks, void* d_counts, void* stream);

/* Same, into HOST memory, synchronous. */
bool horizonator_viewshed(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                          float target_height_m, uint32_t* masks, uint32_t* counts);

/* Per-kernel device times.  While enabled, every render records CUDA events around each of
 * its kernels on the stream it runs on.  horizonator_profile_read() waits for them and reports
 * the MEAN duration in milliseconds per render of: out_ms[0] k_prepare (clear + axis tables),
 * [1] the foreground tiles (k_near: mesh, projection, exact cull; k_raster), [2] k_big of the
 * foreground, [3] the bands of the rest of the mesh (k_tiles, k_blocks, k_mesh, k_raster each, and
 * k_big between bands for zoomed-in views), [4] the last k_big, [5] k_resolve (keys -> image +
 * ranges), over the *renders recorded since the last read.  Profiled renders launch their kernels
 * one by one instead of replaying the captured CUDA graph. */
bool horizonator_profile_enable(const horizonator_context_t* ctx, bool on);
bool horizonator_profile_read(const horizonator_context_t* ctx, float out_ms[6], int* renders);

/* Counters of the most recent render on this context: out[0] = (triangle, sub-box) pairs
 * queued for the large-triangle kernel, out[1] = that queue's capacity, out[2] = kernel
 * launches the render issued, out[3] = CUDA device ordinal, out[4] = triangles that passed
 * the cull and were set up for rasterisation. */
bool horizonator_last_render_stats(const horizonator_context_t* ctx, unsigned int out[5]);

/* Culling counters of the most recent render, collected only while horizonator_profile_enable()
 * is on (all zero otherwise): out[0..3] far-pass tiles looked at / dropped
 * beyond zfar / dropped without a pixel centre in their screen box / dropped as occluded,
 * out[4..7] the same for 4x4-cell blocks (both passes), out[8] blocks whose 32 triangles were
 * projected and tested exactly, out[9] triangles set up, out[10] large-triangle queue entries;
 * out[11..15] reserved (0). */
bool horizonator_render_counters(const horizonator_context_t* ctx, unsigned int out[16]);

#ifdef __cplusplus
}
#endif
