/* horizonator_oracle.h -- TEST INFRASTRUCTURE (oracle).  Not part of the product; only
 * tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may use it.
 *
 * CPU restatement of the reference's render hot path: DEM access (dem.c), the per-render
 * host logic of horizonator-lib.c (move / pan_zoom / set_zextents / render_offscreen incl.
 * the depth->range readback), on top of the GL-pipeline restatement in gl_pipeline.c.
 * Each function cites the reference lines it follows.
 *
 * Pinning: tests/test_oracle.py checks this restatement bit-for-bit against the
 * reference's own dem.c and horizonator-lib.c compiled from /root/reference (oracle/_ref,
 * where horizonator-lib.c runs unmodified on a fake GL whose draw call is gl_pipeline.c),
 * and against the golden vectors in tests/golden/ that were generated from that build.
 * The reference ships no tests or golden vectors of its own.  The rasterisation rules
 * (gl_pipeline.c, F1-F9) restate the OpenGL specification and are pinned against a real GL
 * driver: the unmodified reference on Mesa llvmpipe (oracle/mesa/; tests/test_llvmpipe.py
 * compares this oracle with its recorded and live renders at the north_star tolerances).
 */
#pragma once
#include <stdbool.h>
#include <stdint.h>

#include "gl_pipeline.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct oracle_context oracle_context_t;

/* dem.c:78-243 + horizonator-lib.c:61-680 (offscreen, untextured).  NULL on failure. */
oracle_context_t* oracle_init(float viewer_lat, float viewer_lon, float* viewer_z,
                              int width, int height,
                              int render_radius_cells, float render_radius_m,
                              bool SRTM1, const char* dir_dems);
void oracle_deinit(oracle_context_t* ctx);

bool oracle_move        (oracle_context_t* ctx, float* viewer_z, float lat, float lon); /* lib:691-816 */
bool oracle_pan_zoom    (oracle_context_t* ctx, float az_deg0, float az_deg1);          /* lib:818-836 */
bool oracle_set_zextents(oracle_context_t* ctx, float znear, float zfar,
                         float znear_color, float zfar_color);                          /* lib:864-885 */
bool oracle_render_offscreen(oracle_context_t* ctx, char* image, float* ranges);        /* lib:911-1051 */

/* dem.c:264-309 */
int16_t oracle_dem_sample(const oracle_context_t* ctx, int i, int j);

/* introspection for tests: origin_dem_lon_lat[2], origin_dem_cellij[2], Ndems_ij[2],
 * radius_cells, cells_per_deg -> out[8]; viewer_cell_i, viewer_cell_j, viewer_z,
 * cos_viewer_lat -> outf[4] */
void oracle_get_dem_geometry(const oracle_context_t* ctx, int out[8]);
void oracle_get_viewer(const oracle_context_t* ctx, float outf[4]);

/* opt-in extension, not in the reference: apparent height drop = coefficient * distance^2 (0 = off) */
void oracle_set_curvature(oracle_context_t* ctx, float coefficient);
/* opt-in extension, not in the reference: draw seam-straddling triangles at both edges instead of dropping them */
void oracle_set_seam_wrap(oracle_context_t* ctx, bool on);

/* number of OpenMP threads the draw uses (1 = strictly serial). Default 1. */
void oracle_set_threads(oracle_context_t* ctx, int nthreads);

/* The exact reference of the renderer (tests/test_exact_reference.py, tests/test_gpu_exact.py): visibility keys drawn
 * by glp_draw_keys() from any vertex stage, read back by the code of oracle_render_offscreen().
 * oracle_vertex_stage: this oracle's own vertex stage for the context's (2R)^2 vertices, j outer -> out; returns the
 * seam period (0 without the seam wrap).
 * oracle_read_keys: image and ranges (either may be NULL) of a W x H target of keys, bottom row first, as
 * oracle_render_offscreen() reads them out of its framebuffer for that window and z extents. */
float oracle_vertex_stage(const oracle_context_t* ctx, glp_vtx_t* out);
bool  oracle_read_keys(const uint64_t* keys, int W, int H, float az_deg0, float az_deg1, float znear, float zfar,
                       char* image, float* ranges);

#ifdef __cplusplus
}
#endif
