/* gl_pipeline.h -- TEST INFRASTRUCTURE (oracle).  Not part of the product; only tests/,
 * __graft_entry__.smoke() and bench.py's CPU-baseline legs may use anything under oracle/.
 *
 * CPU restatement of the part of the reference's render path that lives in the OpenGL
 * driver: its three GLSL programs plus the fixed-function stages they run between.
 *
 *   vertex stage     /root/reference/vertex.glsl:30-38,111-162
 *   geometry stage   /root/reference/geometry.glsl:21-35
 *   fragment stage   /root/reference/fragment.glsl:15-16 (untextured branch)
 *   fixed function   state set at /root/reference/horizonator-lib.c:183-185 (depth test,
 *                    back-face cull, clear colour 0,0,1), renderbuffer formats :631,:646,
 *                    viewport :657, clear+draw :896-897; everything else GL defaults.
 *
 * The GL driver itself (Mesa; no version is pinned by the reference, see rpmpackage.spec)
 * is a third-party dependency that is absent from /root/reference.  The fixed-function
 * rules below restate the OpenGL 4.2 core specification (sections 2.14 "coordinate
 * transformations", 3.6.1 "basic polygon rasterization", 4.1.5 "depth buffer test") with
 * the implementation-defined choices written down in gl_pipeline.c.  PINNING: they are
 * checked against a real driver -- the unmodified reference running on Mesa 18.1.9
 * llvmpipe (oracle/mesa/, oracle/_ref/libhorizonator_mesa.so; renders recorded in
 * tests/golden/llvmpipe_*.npz and fullsize_c{1,2}_llvmpipe.npz, compared by
 * tests/test_llvmpipe.py at the north_star tolerances: coverage differs on a handful of
 * pixels per million, range disagreements only on silhouettes).  The host-side logic
 * around them is pinned bit for bit against the reference's own code (oracle/_ref).
 */
#pragma once
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* the uniforms vertex.glsl:8-24 reads on the untextured path */
typedef struct
{
    float viewer_cell_i, viewer_cell_j;
    float viewer_z;
    float DEG_PER_CELL;
    float cos_viewer_lat;
    float az_deg0, az_deg1;
    float aspect;
    float znear, zfar;
    float znear_color, zfar_color;
    /* NOT in the reference (its vertex.glsl:65-88 only estimates the error of ignoring it): opt-in earth
     * curvature + refraction, apparent height drop = curvature * horizontal_distance^2.  0 = the reference. */
    float curvature;
    /* NOT in the reference either (geometry.glsl:15-27 drops them): opt-in, nonzero = draw a triangle that
     * straddles the window's +-pi seam twice, once at each edge of the window. */
    int   seam_wrap;
} glp_uniforms_t;

/* what the vertex stage hands on: gl_Position.xyz (w is 1) and rgb.r */
typedef struct
{
    float x_ndc, y_ndc, z_ndc;
    float r;
} glp_vsout_t;

/* colour: 3 bytes R,G,B per pixel; depth: 24-bit unsigned normalised; both bottom row first
 * (GL window coordinates, y up) */
typedef struct
{
    int       width, height;
    uint8_t*  rgb;   /* width*height*3 */
    uint32_t* z24;   /* width*height   */
} glp_framebuffer_t;

#define GLP_Z24_MAX 0xFFFFFFu

/* one vertex after the vertex stage and the viewport transform (F1): gl_Position.x for the geometry stage, the window
 * coordinates, and the red channel */
typedef struct
{
    float x_ndc;
    float xw, yw, zw;
    float r;
} glp_vtx_t;

/* Visibility key of glp_draw_keys(), one per pixel: the renderer's (horizonator_b200/csrc/hz_device.h) without its
 * epoch bits.  [60:37] q (F7), [36:8] triangle number & GLP_KEY_ID_MASK, [7:0] r8 (F8).  The minimum over a pixel's
 * fragments is GL_LESS in draw order (nearest q, equal q: lowest triangle number); a fragment with q = GLP_Z24_MAX
 * cannot pass GL_LESS against the cleared depth and is dropped. */
#define GLP_KEY_Q_SHIFT 37
#define GLP_KEY_ID_MASK 0x1FFFFFFFull
#define GLP_KEY_CLEAR   0x1FFFFFFFFFFFFFFFull    /* nothing drawn: q = GLP_Z24_MAX */
#define GLP_TILE_CELLS  32                       /* tiles of the level-of-detail rule (HZ_TILE_CELLS) */

void glp_vertex_stage(const glp_uniforms_t* u, float vi, float vj, float vz, glp_vsout_t* out);

int  glp_framebuffer_alloc(glp_framebuffer_t* fb, int width, int height);
void glp_framebuffer_free (glp_framebuffer_t* fb);

/* glClear(COLOR|DEPTH) with clear colour (0,0,1) and clear depth 1.0 */
void glp_clear(glp_framebuffer_t* fb);

/* glDrawElements(GL_TRIANGLES) of ntriangles triangles over nvertices int16 (i,j,z) vertices.
 * indices == NULL selects the reference's dense-grid index pattern
 * (horizonator-lib.c:496-508) for a grid `grid_width` vertices wide, generated on the fly
 * instead of being read from memory.  nthreads<=1: strictly serial, in draw order.
 * nthreads>1: contiguous runs of triangles are drawn into private framebuffers which are
 * then merged in run order with the same strict LESS test; the result is identical to the
 * serial one. */
void glp_draw_triangles(glp_framebuffer_t* fb, const glp_uniforms_t* u,
                        const int16_t* vertices_ijz, int64_t nvertices,
                        const uint32_t* indices, int64_t ntriangles,
                        int grid_width, int nthreads);

/* the vertex stage and the viewport transform of glp_draw_triangles() for nvertices int16 (i,j,z) vertices */
void glp_vertices(const glp_uniforms_t* u, const int16_t* vertices_ijz, int64_t nvertices, int W, int H,
                  glp_vtx_t* vtx, int nthreads);
/* period of x_ndc of the opt-in seam wrap, 0 when it is off */
float glp_seam_period(const glp_uniforms_t* u);

/* Every triangle of the dense grid of N x N vertices vtx[j * N + i], rasterised by the same rules F2-F8 as
 * glp_draw_triangles() (and the seam copies when seam_period > 0), into one visibility key per pixel of a W x H
 * target, bottom row first.  No culling of any kind.  tile_levels == NULL: the reference's mesh.  Otherwise the
 * level of detail l of each tile of GLP_TILE_CELLS x GLP_TILE_CELLS cells, [tj][ti] over ceil((N-1)/32) tiles per
 * side: the tile draws its cells (j, i) with j and i multiples of s = 2^l and at most N-1-s, triangles of vertices s
 * apart, numbered like the cell (j, i) of the dense grid.  Threads draw into private buffers that are merged by min(),
 * so the result does not depend on nthreads.  0 if memory ran out. */
int glp_draw_keys(uint64_t* keys, int W, int H, const glp_vtx_t* vtx, int N, float seam_period,
                  const int8_t* tile_levels, int nthreads);
/* the framebuffer as GL would hold it after drawing those keys' fragments into a cleared one */
void glp_keys_to_framebuffer(const uint64_t* keys, glp_framebuffer_t* fb);

/* glReadPixels(GL_BGR, GL_UNSIGNED_BYTE), pack alignment 1, bottom row first */
void glp_read_bgr(const glp_framebuffer_t* fb, uint8_t* out);
/* glReadPixels(GL_DEPTH_COMPONENT, GL_FLOAT), bottom row first */
void glp_read_depth_float(const glp_framebuffer_t* fb, int x, int y, int w, int h, float* out);

#ifdef __cplusplus
}
#endif
