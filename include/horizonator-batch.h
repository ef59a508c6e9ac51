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

/* Viewshed heights ("above ground level"): for each of n views and each vertex of the loaded square, how far above the
 * ground a point at the vertex must rise for the view to see it; and for every vertex the least of that over the views
 * (how high one may build there and stay hidden from every view).
 *
 * Definition: the views, eye, domain, rays, metres and curvature of the viewshed above (az_deg0 / az_deg1 ignored; no
 * target height).  For a step of a ray that decides vertex v = (i, rint(b)):
 *   - A = (zr - viewer_z) - curvature * d2r and D = sqrt(d2r): the vertex's apparent height and horizontal distance,
 *     exactly the terms the mask's test is built from before target_height_m is added (q = (A + t) / D);
 *   - smax = the largest s of the ray's EARLIER steps (-inf at the first step), as for the mask;
 *   - the step's height e = smax * D - A in fp32, each operation rounded once in that order, then e > 0 ? e : +0
 *     (so -inf, negatives and -0 all become +0).
 *   heights[v] = the least e over all steps of all rays that decide v; the four vertices around the eye are +0; a
 *   vertex that no step decides is +inf.  Every value is >= +0 or +inf and never NaN, so the minimum is taken exactly
 *   and in any order on the 32-bit patterns (hz_kernels.cu: k_viewshed_heights, the mask's own walk;
 *   oracle/viewshed_heights_oracle.c: vs_oracle_r2_heights; the GPU and the oracle agree bit for bit).
 * Relation to the mask: mathematically heights[v] <= t <=> the viewshed at target_height_m = t sees v.  In fp32 the two
 * can differ where t is within rounding of the step's terms (e compares smax * D - A with t, the mask (A + t) / D with
 * smax).  Exactly: isfinite(heights[v]) equals the mask at t = 1e30 (there every decided vertex passes).
 *
 * heights: n x N x N float ([view][j][i]), overwritten;
 * least:   N x N float, least[c] = min(least[c], heights of every view of the call), on the 32-bit patterns (the float
 *          order for values >= +0 and +inf): the caller fills it with +inf once; several calls and several ranks can
 *          fold into one buffer;
 * either may be NULL, not both.  Arguments as for the viewshed: n = 0 does nothing and returns true; n < 0, NULL views,
 * both outputs NULL, an eye outside [0, N-1)^2 or N * N >= 2^32 - 1 return false and write nothing.
 * Sizes: one view's heights are 549 MB at N = 11716 (C2, 150 km of SRTM1), 23 MB at N = 2400 (SRTM3, R = 1200):
 * per-view heights are meant for a few views or small squares; least is the output that scales.  The device call
 * writes per-view heights in place and needs no scratch; without them the walk folds straight into least. */
bool horizonator_viewshed_heights_device(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                                         float* d_heights, float* d_least, void* stream);

/* Same, into HOST memory, synchronous; least is min-folded into the caller's array.  Uses a device copy of least
 * (N x N, allocated on first use) and, for per-view heights, a scratch of at most 64 views and at most 2 GiB (3 views
 * per launch at N = 11716), allocated on first use. */
bool horizonator_viewshed_heights(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                                  float* heights, float* least);

/* Labels of points of interest (POIs): for each of n views and each of m POIs, whether the view sees the POI and where
 * its marker goes -- the rule of the reference's annotator (annotator.c:280-348), which the command-line tool's
 * --labels output follows (cli/horizonator-standalone.c, write_labels()), evaluated on the GPU for whole batches.
 *
 * Rule, per (view, POI):
 *   - Projection: horizonator_project() in double with lat_viewer = (double)view.lat, lon_viewer = (double)view.lon,
 *     cos_lat_viewer = cos(lat_viewer * pi / 180) (computed on the host per view), ele_viewer = the eye height as
 *     horizonator_move() computes it (automatic when viewer_z < 0), az_rad0/1 = (double)az_deg0/1 * pi / 180, and the
 *     context's W and H.  The GPU evaluates the same source operator for operator (no fused multiply-adds); only
 *     atan2() may differ from the host's in the last bit.
 *   - Gates: 500 m <= range <= 100 km, and lround(x) in [0, W).
 *   - Vertical search, at column col = lround(x): for d = -6 .. 5 in turn: skip d while y + d < 0, stop once
 *     y + d >= H; row r = lround(y) + d, skipped outside [0, H); skip rows whose rendered range is <= 0 (sky); the
 *     error is |range - rendered range|: keep the first d with the smallest error so far and stop as soon as an error
 *     is not smaller than the best.  The POI is visible iff the best error is below 500 m.
 *   - The rendered ranges are the render's own, bit-identical to what the range image of the same render holds
 *     (they are read from the visibility buffer and converted exactly as the range image is).
 * Output, horizonator_label_t, each double rounded to float once:
 *   - horizonator_project() fails (outside the window): all four fields -1;
 *   - otherwise x and range_m are set; y is the projected y plus the search offset when visible, the projected y
 *     otherwise; range_rendered_m is the matched rendered range when visible, -1 otherwise: visible <=> > 0.
 * Known limits:
 *   - A window of exactly 360 degrees (az_deg1 - az_deg0 == 360 in double, e.g. -180 .. 180) places no POI: the
 *     reference's horizonator_project() unwraps its width to 0 and fails for every point, so every label is -1.
 *     A window a fraction of a degree narrower works.
 *   - The projection is the reference's flat-earth one.  With horizonator_set_earth_curvature() on, distant terrain is
 *     drawn lower than horizonator_project() puts the POIs on it, so a POI far enough away sits above the terrain as
 *     drawn and the +-6-row search can miss it.  The labels do not correct for that.
 *   - The labels take n * m * 16 bytes.  For the host-memory call, from roughly 50 k POIs per view copying them, not
 *     rendering, is what limits the rate (an estimate from the measured device->host copy rate, not a measurement).
 */
typedef struct { double lat, lon, ele; } horizonator_poi_t;                     /* 24 bytes; ele in metres */
typedef struct { float x, y, range_m, range_rendered_m; } horizonator_label_t;  /* 16 bytes */

/* Renders the n views exactly as horizonator_render_batch_device() does (same chunks, the context's z extents, size
 * and opt-in modes) and writes d_labels[k * m + i] for view k and POI i.  views: host memory; d_pois (8-byte aligned)
 * and d_labels (16-byte aligned): DEVICE memory.  d_images / d_ranges as in horizonator_render_batch_device(), either
 * or both may be NULL: with both NULL no panorama is written at all, only the labels.  Stream as for the batch render.
 * n == 0 or m == 0: nothing is done, true.  n < 0, m < 0, or NULL views / POIs / labels otherwise: false, nothing is
 * written. */
bool horizonator_annotate_batch_device(const horizonator_context_t* ctx,
                                       int n, const horizonator_view_t* views,
                                       int m, const horizonator_poi_t* d_pois,
                                       horizonator_label_t* d_labels,
                                       void* d_images, void* d_ranges, void* stream);

/* Same with pois and labels in HOST memory, synchronous; no panorama is written, and only the n * m labels cross the
 * bus (into page-locked memory by DMA; see horizonator_host_alloc()). */
bool horizonator_annotate_batch(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                                int m, const horizonator_poi_t* pois, horizonator_label_t* labels);

/* Skylines, and their match against an observed skyline: for each of n views, the topmost terrain pixel of every
 * column, and how well the skyline traced from a photo fits that view at every heading -- the search for where a photo
 * was taken and which way it looks, over batches of candidate eyes, on the GPU.
 *
 * Render: each view is rendered exactly as horizonator_render_batch_device() renders it (the same chunks, captured
 * graphs, the context's z extents and size, and the same opt-in modes: earth curvature, seam wrap, level of detail);
 * terrain beyond zfar is sky, as in the image.  No image and no range image is written.
 * Rows and range: rows[k * W + c] is the image row (0 = top) of the topmost terrain pixel of column c of view k, or -1
 * if the column is all sky; range[k * W + c] is that pixel's range, or -1.  Both are bit-identical to
 * horizonator_horizon_profile_device() applied to the range image of the same render.
 * Samples: a sample (dx, y) says that dx columns right of the heading column the observed skyline lies at pixel
 * coordinate y (pixel centres at integer y, 0 = top: the y of horizonator_project()).  From angles: with
 * p = (az_deg1 - az_deg0) / W degrees per column, a skyline point rel_az_deg right of the heading and el_deg above the
 * horizontal is dx = rint(rel_az_deg / p), y = (H - 1) / 2 - el_deg / p, evaluated in double and rounded to float once
 * -- horizonator_project()'s y at the same angle, since x and y share one angular scale.
 * Score, for view k and every heading column h in [0, W), whose heading is the azimuth of its centre,
 * az_deg0 + (h + 0.5) * p:
 *   - c_i = h + dx_i; with `wrap` taken modulo W (non-negative; meant for full-circle windows), without it a c_i
 *     outside [0, W) is missing;
 *   - d_i = fminf(fabsf(((float)s - 0.5f) - y_i), clip_rows) with s = rows[k][c_i] (the rendered skyline's edge lies
 *     half a row above its topmost terrain pixel); an all-sky (s = -1) or missing column gives d_i = clip_rows;
 *   - scores[k * W + h] = (d_0 + d_1 + ... + d_{m-1}) / (float)m, the fp32 sum in that order, every operation rounded
 *     once: the scores are reproducible exactly.  0 is a perfect fit; clip_rows is the worst.
 * Arguments: views in host memory; any of rows, range and scores may be NULL, not all three; scores need m >= 1, the
 * samples and a finite clip_rows > 0, and an image at most 32767 rows high and (shared memory) about 110 000 columns
 * wide; without scores m, samples, clip_rows and wrap are ignored.  n == 0: nothing is done, true.  Bad arguments:
 * false, nothing is written.  Each output takes n * W * 4 bytes.
 */
typedef struct { int32_t dx; float y; } horizonator_skyline_sample_t;     /* 8 bytes */

/* d_rows, d_range, d_scores (4-byte aligned) and d_samples (8-byte aligned): DEVICE memory.  Stream as for the batch
 * render. */
bool horizonator_skyline_match_device(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                                      int* d_rows, float* d_range,
                                      int m, const horizonator_skyline_sample_t* d_samples,
                                      float clip_rows, bool wrap, float* d_scores, void* stream);

/* Same with everything in HOST memory, synchronous; only the n * W * (4 to 12) bytes asked for cross the bus (into
 * page-locked memory by DMA; see horizonator_host_alloc()). */
bool horizonator_skyline_match(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                               int* rows, float* range,
                               int m, const horizonator_skyline_sample_t* samples,
                               float clip_rows, bool wrap, float* scores);

/* What is at this pixel: for each of n views and each of m pixels (or every pixel), the ground point the pixel shows --
 * its latitude, longitude, height and distance, the triangle of the DEM mesh it lies on, and the pixel's range -- read
 * from the triangle number each visibility key of the render holds.
 *
 * Render: each view is rendered exactly as horizonator_render_batch_device() renders it (the same chunks, captured
 * graphs, the context's z extents and size, and the same opt-in modes: earth curvature, seam wrap, level of detail).
 * Images and range images are written only where d_images / d_ranges are given.
 * DEM geometry (dem.h): mesh vertex (i, j) -- column i east, row j north, as horizonator_download_mosaic() indexes the
 * square -- lies at
 *     lon = origin_dem_lon_lat[0] + (origin_dem_cellij[0] + i) / cells_per_deg
 *     lat = origin_dem_lon_lat[1] + (origin_dem_cellij[1] + j) / cells_per_deg
 * evaluated in double with i, j real (the fields are those of ctx->dems).
 * Per pixel (x, y) of view k (x column, y row, 0 = top, as the image):
 *   - The key at GL row H-1-y, column x decides.  Sky -- nothing of this render drawn there, or (x, y) outside the
 *     image -- gives triangle = 0xFFFFFFFF, range_m = -1 and lat = lon = ele_m = distance_m = NaN.
 *   - range_m: the pixel's range, bit-identical to the range image of the same render.
 *   - triangle: the number of the triangle drawn there, as the reference numbers them (horizonator-lib.c:496-508:
 *     2 * (j * (N - 1) + i) + half, N = 2 * radius_cells, (j, i) its first vertex), with the level of detail of the
 *     band it was drawn in in bits [30:29] (0 without horizonator_set_lod(); level l: vertices 2^l cells apart, half 0
 *     = (j,i), (j+s,i+s), (j+s,i) and half 1 = (j,i), (j,i+s), (j+s,i+s), s = 2^l).  The level is that of the band of
 *     rings of 32x32-cell tiles around the eye's tile that holds the tile of (j, i); bands do not overlap, so it is
 *     unique.
 *   - Ground point: the three vertices' window positions as the renderer computes them before snapping (float,
 *     vertex.glsl and the viewport transform; with the seam wrap the copy of the triangle whose x-range holds the pixel
 *     centre); the barycentric weights (b0, b1, b2) of the pixel centre (cx, cy) = (x + 0.5, H - 1 - y + 0.5) from them,
 *     in double, not clamped:
 *         d  = (x1 - x0) * (y2 - y0) - (x2 - x0) * (y1 - y0)
 *         b1 = ((cx - x0) * (y2 - y0) - (x2 - x0) * (cy - y0)) / d
 *         b2 = ((x1 - x0) * (cy - y0) - (cx - x0) * (y1 - y0)) / d
 *         b0 = 1 - b1 - b2
 *     and with S(a) = b0 * a0 + b1 * a1 + b2 * a2: i = S(vertex columns), j = S(vertex rows) -> lat, lon by the DEM
 *     geometry; ele_m = S(terrain heights) (the true height, not the apparent one of the opt-in curvature);
 *     distance_m = sqrt(E * E + N * N) with E, N = S of the vertices' metres east / north of the eye as the renderer
 *     computes them (float, vertex.glsl:128-130).  All in double, every operation rounded once in the order written;
 *     ele_m and distance_m rounded to float once.
 * Limits: the point is the screen-space interpolation GL gives an attribute over the triangle (what the reference's
 * texture mode does with its per-vertex texture coordinate, vertex.glsl:116-126), not the intersection of the pixel's
 * ray with the surface.  The rasteriser decides coverage on positions snapped to 1/256 pixel, so at a silhouette a
 * weight can lie up to about 1/256 pixel's worth outside [0, 1].  Whole-image output takes H * W * 32 bytes per view
 * (69 MB at 3600 x 600).
 * Arguments: views in host memory.  pixels (8-byte aligned): [n][m]; NULL: every pixel, the output is then [n][H][W]
 * in image order and m (>= 0) is not used.  ground (8-byte aligned): [n][m] or [n][H][W].  n == 0, or m == 0 with
 * pixels given: nothing is done, true.  n < 0, m < 0, NULL views or ground otherwise, or misaligned pointers: false,
 * nothing is written. */
typedef struct { int32_t x, y; } horizonator_pixel_t;     /* 8 bytes: column, row (0 = top), as the image */
typedef struct
{
    double   lat, lon;
    float    ele_m, range_m, distance_m;
    uint32_t triangle;
} horizonator_ground_t;                                    /* 32 bytes */

/* d_pixels, d_ground: DEVICE memory; d_images / d_ranges as in horizonator_render_batch_device(), either or both may be
 * NULL.  Stream as for the batch render. */
bool horizonator_pick_batch_device(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                                   int m, const horizonator_pixel_t* d_pixels, horizonator_ground_t* d_ground,
                                   void* d_images, void* d_ranges, void* stream);

/* Same with pixels and ground in HOST memory, synchronous; no panorama is written, and only the ground points cross
 * the bus (into page-locked memory by DMA; see horizonator_host_alloc()).  Unlike horizonator_pick() (horizonator.h),
 * which unprojects one pixel of the context's last render treating its depth as a horizontal distance, this reads the
 * exact triangle. */
bool horizonator_pick_batch(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                            int m, const horizonator_pixel_t* pixels, horizonator_ground_t* ground);

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
 * projected and tested exactly, out[9] triangles set up, out[10] large-triangle queue entries,
 * out[11] tiles and blocks found occluded from the span grid alone, without reading their keys
 * (counted in out[3] and out[7] too), out[12] 8x8 blocks of the visibility buffer whose span
 * grid words were recomputed; out[13..15] reserved (0). */
bool horizonator_render_counters(const horizonator_context_t* ctx, unsigned int out[16]);

#ifdef __cplusplus
}
#endif
