/* gl_pipeline.c -- TEST INFRASTRUCTURE (oracle); see gl_pipeline.h for scope and pinning.
 *
 * All arithmetic that the reference does in GLSL `float` is done here in C `float`, one IEEE
 * operation per source operator, left to right, no fused multiply-add (build with
 * -ffp-contract=off).  Transcendentals are the C library's (atan2f, sqrtf).
 *
 * Implementation-defined choices of the fixed-function stages (GL 4.2 core leaves these to
 * the driver; the values follow common software rasterisers and are the contract the CUDA
 * path is tested against):
 *   F1  viewport transform: xw = x_ndc*(W/2) + W/2, yw likewise, zw = z_ndc*0.5 + 0.5.
 *   F2  window positions are snapped to 1/256 pixel in float: t = xw*256;
 *       X = |t| < 2^23 ? floorf(t + 0.5f) : t   (beyond 2^23 a float is already an integer).
 *   F3  facing and coverage use exact integer edge functions on the snapped positions;
 *       counter-clockwise (area > 0, y up) is front; back faces and zero-area are culled.
 *   F4  a pixel is covered iff its centre (px+.5, py+.5) is strictly inside, or lies on an
 *       edge that runs downwards (dy<0) or is horizontal running leftwards (dy==0, dx<0).
 *       Two triangles sharing an edge therefore never both produce the pixel.
 *   F5  clipping to the view volume: w is 1 for every vertex, so interpolation is affine and
 *       clipping is applied per fragment: outside the viewport or zw outside [0,1] => dropped.
 *       A triangle with a vertex beyond +-2^21 pixels (or a non-finite one) is dropped
 *       (keeps the 64-bit edge functions on 1/256-pixel coordinates free of overflow).
 *   F6  zw and the red channel are interpolated as planes through the UNSNAPPED float
 *       vertices, anchored at the triangle's first vertex, evaluated at the pixel centre.
 *       The pixel centre can lie up to 1/256 pixel outside the unsnapped triangle, so the
 *       plane is extrapolated a little; across a sliver thinner than that the extrapolation
 *       is unbounded.  The interpolated zw is therefore limited to the range of the three
 *       vertex values widened by 4x its own extent on either side (reached only by slivers
 *       thinner than about 1/1000 pixel, where the value is an artefact anyway).
 *   F7  GL_DEPTH_COMPONENT renderbuffer = 24-bit unsigned normalised: q = floor(zw*(2^24-1)+.5);
 *       test GL_LESS on q against the stored q, cleared to 2^24-1; read back as float(q/(2^24-1)).
 *   F8  GL_RGB renderbuffer = 8-bit unsigned normalised: c8 = floor(clamp(c,0,1)*255 + .5).
 *   F9  GLSL round() (vertex.glsl:37) rounds halfway cases to even.
 */
#include "gl_pipeline.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ---------------------------------------------------------------- vertex stage */

static const float Rearth = 6371000.0f;         /* vertex.glsl:30 */
static const float pi     = 3.14159265358979f;  /* vertex.glsl:31 */

/* vertex.glsl:34-38 */
static float unwrap_near_rad(float x, float near)
{
    float d = (x - near) / (2.f * pi);
    return (d - rintf(d)) * 2.f * pi + near;    /* F9 */
}

/* GLSL radians(): multiplication by the float constant pi/180 */
static float glsl_radians(float deg) { return deg * 0.017453292519943295f; }

/* vertex.glsl:111-162, the live branch, NtilesX == 0 */
void glp_vertex_stage(const glp_uniforms_t* u, float vi, float vj, float vz, glp_vsout_t* out)
{
    float i = vi, j = vj;

    float en_x = (i - u->viewer_cell_i) * u->DEG_PER_CELL * Rearth * pi / 180.f * u->cos_viewer_lat;
    float en_y = (j - u->viewer_cell_j) * u->DEG_PER_CELL * Rearth * pi / 180.f;
    float enh_z = vz - u->viewer_z - u->curvature * (en_x * en_x + en_y * en_y);   /* curvature == 0: the reference */

    float distance_ne = sqrtf(en_x * en_x + en_y * en_y);       /* length(en)      :133 */
    float az_rad      = atan2f(en_x, en_y);                     /* atan(en.x,en.y) :134 */

    float az_rad0 = glsl_radians(u->az_deg0);
    float az_rad1 = glsl_radians(u->az_deg1);
    az_rad1 = unwrap_near_rad(az_rad1 - az_rad0, pi) + az_rad0; /* :143 */

    float az_rad_center = (az_rad0 + az_rad1) / 2.f;            /* :146 */
    az_rad = unwrap_near_rad(az_rad, az_rad_center);            /* :148 */

    float az_ndc_per_rad = 2.0f / (az_rad1 - az_rad0);          /* :150 */

    out->x_ndc = (az_rad - az_rad_center) * az_ndc_per_rad;                   /* :152 */
    out->y_ndc = atan2f(enh_z, distance_ne) * u->aspect * az_ndc_per_rad;     /* :153 */
    float length_enh = sqrtf(en_x * en_x + en_y * en_y + enh_z * enh_z);
    out->z_ndc = (length_enh - u->znear) / (u->zfar - u->znear) * 2.f - 1.f;  /* :155 */

    out->r = fmaxf(fminf((distance_ne - u->znear_color) / (u->zfar_color - u->znear_color),
                         1.0f), 0.0f);                                        /* :159-160 */
}

/* ---------------------------------------------------------------- framebuffer */

int glp_framebuffer_alloc(glp_framebuffer_t* fb, int width, int height)
{
    fb->width = width; fb->height = height;
    fb->rgb = (uint8_t*) malloc((size_t)width * height * 3);
    fb->z24 = (uint32_t*)malloc((size_t)width * height * sizeof(uint32_t));
    if(!fb->rgb || !fb->z24) { glp_framebuffer_free(fb); return 0; }
    return 1;
}
void glp_framebuffer_free(glp_framebuffer_t* fb)
{
    free(fb->rgb); free(fb->z24);
    fb->rgb = NULL; fb->z24 = NULL;
}

/* horizonator-lib.c:185 glClearColor(0,0,1,0); :896 glClear; clear depth default 1.0 */
void glp_clear(glp_framebuffer_t* fb)
{
    size_t n = (size_t)fb->width * fb->height;
    for(size_t p = 0; p < n; p++)
    {
        fb->rgb[3*p+0] = 0; fb->rgb[3*p+1] = 0; fb->rgb[3*p+2] = 255;
        fb->z24[p] = GLP_Z24_MAX;
    }
}

void glp_read_bgr(const glp_framebuffer_t* fb, uint8_t* out)
{
    size_t n = (size_t)fb->width * fb->height;
    for(size_t p = 0; p < n; p++)
    {
        out[3*p+0] = fb->rgb[3*p+2];
        out[3*p+1] = fb->rgb[3*p+1];
        out[3*p+2] = fb->rgb[3*p+0];
    }
}

void glp_read_depth_float(const glp_framebuffer_t* fb, int x, int y, int w, int h, float* out)
{
    const double scale = 1.0 / (double)GLP_Z24_MAX;              /* F7 */
    for(int yy = 0; yy < h; yy++)
        for(int xx = 0; xx < w; xx++)
            out[(size_t)yy * w + xx] =
                (float)((double)fb->z24[(size_t)(y + yy) * fb->width + (x + xx)] * scale);
}

/* ---------------------------------------------------------------- primitive stages */

#define SUBPIXEL   256
#define GUARD_PX   2097152.0f   /* 2^21 (F5) */

static inline int64_t snap(float a)                                          /* F2 */
{
    float t = a * (float)SUBPIXEL;
    if(fabsf(t) < 8388608.0f) t = floorf(t + 0.5f);
    return (int64_t)t;
}

/* Where draw_one writes a fragment.  zr != NULL: (q<<8)|r8 per pixel under GL_LESS, so a private buffer is one word
 * per pixel.  Otherwise keys: the visibility key of triangle `id` (see GLP_KEY_Q_SHIFT), kept where it is the
 * minimum. */
typedef struct
{
    uint32_t* zr;
    uint64_t* keys;
    uint64_t  id;
} glp_target_t;

static inline void
draw_one(const glp_target_t* tg, int W, int H, const glp_vtx_t* v0, const glp_vtx_t* v1, const glp_vtx_t* v2, float seam_period)
{
    /* geometry.glsl:21-27 */
    float xmax = fmaxf(fmaxf(v0->x_ndc, v1->x_ndc), v2->x_ndc);
    float xmin = fminf(fminf(v0->x_ndc, v1->x_ndc), v2->x_ndc);
    if(xmax - xmin > 0.5f)
    {
        /* opt-in extension (seam_period > 0; the reference stops here): the triangle with its left-hand vertices
         * moved one period of x_ndc to the right, and that moved one period to the left */
        if(seam_period > 0.0f)
        {
            const float halfW = 0.5f * (float)W;
            for(int copy = 1; copy <= 2; copy++)
            {
                glp_vtx_t c[3] = { *v0, *v1, *v2 };
                for(int k = 0; k < 3; k++)
                {
                    if(c[k].x_ndc < 0.0f) c[k].x_ndc += seam_period;
                    if(copy == 2) c[k].x_ndc -= seam_period;
                    c[k].xw = c[k].x_ndc * halfW + halfW;
                }
                draw_one(tg, W, H, &c[0], &c[1], &c[2], 0.0f);
            }
        }
        return;
    }

    /* F5 guard band; also rejects NaN/Inf */
    if(!(fabsf(v0->xw) < GUARD_PX && fabsf(v0->yw) < GUARD_PX &&
         fabsf(v1->xw) < GUARD_PX && fabsf(v1->yw) < GUARD_PX &&
         fabsf(v2->xw) < GUARD_PX && fabsf(v2->yw) < GUARD_PX)) return;

    const int64_t X0 = snap(v0->xw), Y0 = snap(v0->yw);
    const int64_t X1 = snap(v1->xw), Y1 = snap(v1->yw);
    const int64_t X2 = snap(v2->xw), Y2 = snap(v2->yw);

    /* F3: GL_CULL_FACE with glFrontFace(GL_CCW), glCullFace(GL_BACK) defaults */
    const int64_t area = (X1 - X0) * (Y2 - Y0) - (X2 - X0) * (Y1 - Y0);
    if(area <= 0) return;

    /* pixels whose centre (SUBPIXEL*p + SUBPIXEL/2) can lie inside the snapped bounding box */
    int64_t bx0 = X0 < X1 ? X0 : X1; if(X2 < bx0) bx0 = X2;
    int64_t bx1 = X0 > X1 ? X0 : X1; if(X2 > bx1) bx1 = X2;
    int64_t by0 = Y0 < Y1 ? Y0 : Y1; if(Y2 < by0) by0 = Y2;
    int64_t by1 = Y0 > Y1 ? Y0 : Y1; if(Y2 > by1) by1 = Y2;
    /* ceil((b0 - 128)/256) and floor((b1 - 128)/256) with arithmetic shifts */
    int64_t px0 = (bx0 - SUBPIXEL/2 + SUBPIXEL - 1) >> 8, px1 = (bx1 - SUBPIXEL/2) >> 8;
    int64_t py0 = (by0 - SUBPIXEL/2 + SUBPIXEL - 1) >> 8, py1 = (by1 - SUBPIXEL/2) >> 8;
    if(px0 < 0) px0 = 0;
    if(py0 < 0) py0 = 0;
    if(px1 > W - 1) px1 = W - 1;
    if(py1 > H - 1) py1 = H - 1;
    if(px0 > px1 || py0 > py1) return;

    /* F6: planes through the unsnapped float vertices, anchored at v0 */
    const float ax = v1->xw - v0->xw, ay = v1->yw - v0->yw;
    const float bx = v2->xw - v0->xw, by = v2->yw - v0->yw;
    const float det = ax * by - bx * ay;
    const float inv = 1.0f / det;
    const float az = v1->zw - v0->zw, bz = v2->zw - v0->zw;
    const float ar = v1->r  - v0->r,  br = v2->r  - v0->r;
    const float dzdx = (az * by - bz * ay) * inv;
    const float dzdy = (bz * ax - az * bx) * inv;
    const float drdx = (ar * by - br * ay) * inv;
    const float drdy = (br * ax - ar * bx) * inv;
    const float zw_min = fminf(fminf(v0->zw, v1->zw), v2->zw);
    const float zw_max = fmaxf(fmaxf(v0->zw, v1->zw), v2->zw);
    const float zw_lo = zw_min - 4.0f * (zw_max - zw_min);
    const float zw_hi = zw_max + 4.0f * (zw_max - zw_min);

    /* F4: edge a->b owns its boundary iff dy<0 or (dy==0 and dx<0) */
    const int64_t e0dx = X1 - X0, e0dy = Y1 - Y0;
    const int64_t e1dx = X2 - X1, e1dy = Y2 - Y1;
    const int64_t e2dx = X0 - X2, e2dy = Y0 - Y2;
    const int64_t bias0 = (e0dy < 0 || (e0dy == 0 && e0dx < 0)) ? 0 : 1;
    const int64_t bias1 = (e1dy < 0 || (e1dy == 0 && e1dx < 0)) ? 0 : 1;
    const int64_t bias2 = (e2dy < 0 || (e2dy == 0 && e2dx < 0)) ? 0 : 1;

    for(int64_t py = py0; py <= py1; py++)
    {
        const int64_t Py = py * SUBPIXEL + SUBPIXEL/2;
        for(int64_t px = px0; px <= px1; px++)
        {
            const int64_t Px = px * SUBPIXEL + SUBPIXEL/2;
            const int64_t E0 = e0dx * (Py - Y0) - e0dy * (Px - X0);
            const int64_t E1 = e1dx * (Py - Y1) - e1dy * (Px - X1);
            const int64_t E2 = e2dx * (Py - Y2) - e2dy * (Px - X2);
            if(E0 < bias0 || E1 < bias1 || E2 < bias2) continue;

            const float cx = (float)px + 0.5f, cy = (float)py + 0.5f;
            const float ddx = cx - v0->xw, ddy = cy - v0->yw;
            float zw = v0->zw + (dzdx * ddx + dzdy * ddy);
            zw = fminf(fmaxf(zw, zw_lo), zw_hi);                            /* F6 */
            if(!(zw >= 0.0f && zw <= 1.0f)) continue;                       /* F5 */

            const uint32_t q = (uint32_t)((double)zw * (double)GLP_Z24_MAX + 0.5);   /* F7 */
            const size_t p = (size_t)py * W + px;
            if(tg->zr ? !(q < (tg->zr[p] >> 8))                             /* GL_LESS */
                      : (q >= GLP_Z24_MAX || q > (uint32_t)(tg->keys[p] >> GLP_KEY_Q_SHIFT))) continue;

            float r = v0->r + (drdx * ddx + drdy * ddy);                    /* fragment.glsl:16 */
            r = fmaxf(fminf(r, 1.0f), 0.0f);
            const uint32_t r8 = (uint32_t)(r * 255.0f + 0.5f);              /* F8 */
            if(tg->zr) tg->zr[p] = (q << 8) | r8;
            else
            {
                const uint64_t key = ((uint64_t)q << GLP_KEY_Q_SHIFT) | (tg->id << 8) | r8;
                if(key < tg->keys[p]) tg->keys[p] = key;
            }
        }
    }
}

static inline void
triangle_indices(const uint32_t* indices, int64_t t, int gw, int64_t* i0, int64_t* i1, int64_t* i2)
{
    if(indices)
    {
        *i0 = indices[3*t+0]; *i1 = indices[3*t+1]; *i2 = indices[3*t+2];
        return;
    }
    /* horizonator-lib.c:496-508 */
    const int64_t cell = t >> 1;
    const int64_t j = cell / (gw - 1), i = cell % (gw - 1);
    *i0 = j * gw + i;
    if((t & 1) == 0) { *i1 = (j + 1) * gw + (i + 1); *i2 = (j + 1) * gw + i;       }
    else             { *i1 = j * gw + (i + 1);       *i2 = (j + 1) * gw + (i + 1); }
}

/* period of x_ndc for the opt-in seam wrap: az_ndc_per_rad (vertex.glsl:139-150) * 2*pi; 0 without it */
float glp_seam_period(const glp_uniforms_t* u)
{
    if(!u->seam_wrap) return 0.0f;
    float az_rad0 = glsl_radians(u->az_deg0), az_rad1 = glsl_radians(u->az_deg1);
    az_rad1 = unwrap_near_rad(az_rad1 - az_rad0, pi) + az_rad0;
    return 2.0f / (az_rad1 - az_rad0) * 2.f * pi;
}

void glp_vertices(const glp_uniforms_t* u, const int16_t* vertices_ijz, int64_t nvertices, int W, int H,
                  glp_vtx_t* vtx, int nthreads)
{
    const float halfW = 0.5f * (float)W, halfH = 0.5f * (float)H;
    #pragma omp parallel for num_threads(nthreads < 1 ? 1 : nthreads) schedule(static)
    for(int64_t v = 0; v < nvertices; v++)
    {
        glp_vsout_t o;
        /* GL_SHORT, not normalised (horizonator-lib.c:424): the shader sees float(int16) */
        glp_vertex_stage(u, (float)vertices_ijz[3*v+0], (float)vertices_ijz[3*v+1],
                         (float)vertices_ijz[3*v+2], &o);
        vtx[v].x_ndc = o.x_ndc;
        vtx[v].xw = o.x_ndc * halfW + halfW;     /* F1 */
        vtx[v].yw = o.y_ndc * halfH + halfH;
        vtx[v].zw = o.z_ndc * 0.5f + 0.5f;
        vtx[v].r  = o.r;
    }
}

void glp_draw_triangles(glp_framebuffer_t* fb, const glp_uniforms_t* u,
                        const int16_t* vertices_ijz, int64_t nvertices,
                        const uint32_t* indices, int64_t ntriangles,
                        int grid_width, int nthreads)
{
    const int W = fb->width, H = fb->height;
    if(nthreads < 1) nthreads = 1;

    glp_vtx_t* vtx = (glp_vtx_t*)malloc((size_t)nvertices * sizeof(glp_vtx_t));
    if(!vtx) return;
    glp_vertices(u, vertices_ijz, nvertices, W, H, vtx, nthreads);
    const float seam_period = glp_seam_period(u);

    const size_t npix = (size_t)W * H;

    /* the shared target starts from the framebuffer's current contents */
    uint32_t* target = (uint32_t*)malloc(npix * sizeof(uint32_t));
    for(size_t p = 0; p < npix; p++) target[p] = (fb->z24[p] << 8) | fb->rgb[3*p+0];
    /* colour of pixels never touched by this draw is kept as is (see the write-back) */

    if(nthreads == 1)
    {
        const glp_target_t tg = { target, NULL, 0 };
        for(int64_t t = 0; t < ntriangles; t++)
        {
            int64_t i0, i1, i2;
            triangle_indices(indices, t, grid_width, &i0, &i1, &i2);
            draw_one(&tg, W, H, &vtx[i0], &vtx[i1], &vtx[i2], seam_period);
        }
    }
    else
    {
        uint32_t** priv = (uint32_t**)calloc(nthreads, sizeof(uint32_t*));
        #pragma omp parallel num_threads(nthreads)
        {
#ifdef _OPENMP
            const int tid = omp_get_thread_num(), nt = omp_get_num_threads();
#else
            const int tid = 0, nt = 1;
#endif
            uint32_t* mine = (uint32_t*)malloc(npix * sizeof(uint32_t));
            for(size_t p = 0; p < npix; p++) mine[p] = (GLP_Z24_MAX << 8);
            priv[tid] = mine;
            const glp_target_t tg = { mine, NULL, 0 };
            const int64_t t0 = ntriangles * tid / nt, t1 = ntriangles * (tid + 1) / nt;
            for(int64_t t = t0; t < t1; t++)
            {
                int64_t i0, i1, i2;
                triangle_indices(indices, t, grid_width, &i0, &i1, &i2);
                draw_one(&tg, W, H, &vtx[i0], &vtx[i1], &vtx[i2], seam_period);
            }
        }
        /* merge in draw order with the same strict LESS */
        #pragma omp parallel for num_threads(nthreads) schedule(static)
        for(size_t p = 0; p < npix; p++)
        {
            uint32_t cur = target[p];
            for(int k = 0; k < nthreads; k++)
                if(priv[k] && (priv[k][p] >> 8) < (cur >> 8)) cur = priv[k][p];
            target[p] = cur;
        }
        for(int k = 0; k < nthreads; k++) free(priv[k]);
        free(priv);
    }

    for(size_t p = 0; p < npix; p++)
        if((target[p] >> 8) < fb->z24[p])
        {
            fb->z24[p]     = target[p] >> 8;
            fb->rgb[3*p+0] = (uint8_t)(target[p] & 0xFF);   /* rgb = (r,0,0): vertex.glsl:159-162 */
            fb->rgb[3*p+1] = 0;
            fb->rgb[3*p+2] = 0;
        }

    free(target);
    free(vtx);
}

int glp_draw_keys(uint64_t* keys, int W, int H, const glp_vtx_t* vtx, int N, float seam_period,
                  const int8_t* tile_levels, int nthreads)
{
    if(nthreads < 1) nthreads = 1;
    const size_t npix = (size_t)W * H;
    const int nt = (N - 1 + GLP_TILE_CELLS - 1) / GLP_TILE_CELLS;
    uint64_t** priv = (uint64_t**)calloc(nthreads, sizeof(uint64_t*));
    if(!priv) return 0;
    int ok = 1;
    #pragma omp parallel num_threads(nthreads)
    {
#ifdef _OPENMP
        const int tid = omp_get_thread_num();
#else
        const int tid = 0;
#endif
        uint64_t* mine = (uint64_t*)malloc(npix * sizeof(uint64_t));
        if(!mine) ok = 0;
        else for(size_t p = 0; p < npix; p++) mine[p] = GLP_KEY_CLEAR;
        priv[tid] = mine;
        #pragma omp for schedule(dynamic, 1)
        for(int tj = 0; tj < nt; tj++)
        {
            if(!mine) continue;
            for(int ti = 0; ti < nt; ti++)
            {
                const int l = tile_levels ? tile_levels[(size_t)tj * nt + ti] : 0, s = 1 << l;
                /* the last (N - 1) mod s cells of a row or column are not drawn at level l */
                const int jend = GLP_TILE_CELLS * (tj + 1) < N - s ? GLP_TILE_CELLS * (tj + 1) : N - s;
                const int iend = GLP_TILE_CELLS * (ti + 1) < N - s ? GLP_TILE_CELLS * (ti + 1) : N - s;
                for(int j = GLP_TILE_CELLS * tj; j < jend; j += s)
                    for(int i = GLP_TILE_CELLS * ti; i < iend; i += s)
                    {
                        const glp_vtx_t* a = vtx + (size_t)j * N + i;             /* (j, i) */
                        const glp_vtx_t* b = a + s;                               /* (j, i+s) */
                        const glp_vtx_t* c = a + (size_t)s * N;                   /* (j+s, i) */
                        const glp_vtx_t* d = c + s;                               /* (j+s, i+s) */
                        const uint64_t cell = (uint64_t)j * (uint64_t)(N - 1) + (uint64_t)i;
                        /* horizonator-lib.c:496-508 with vertices s apart: (j,i),(j+s,i+s),(j+s,i) and (j,i),(j,i+s),(j+s,i+s) */
                        const glp_target_t t0 = { NULL, mine, (2 * cell) & GLP_KEY_ID_MASK };
                        const glp_target_t t1 = { NULL, mine, (2 * cell + 1) & GLP_KEY_ID_MASK };
                        draw_one(&t0, W, H, a, d, c, seam_period);
                        draw_one(&t1, W, H, a, b, d, seam_period);
                    }
            }
        }
    }
    if(ok)
    {
        /* the minimum over all fragments: the order of the triangles, and so the number of threads, cannot matter */
        #pragma omp parallel for num_threads(nthreads) schedule(static)
        for(size_t p = 0; p < npix; p++)
        {
            uint64_t cur = GLP_KEY_CLEAR;
            for(int k = 0; k < nthreads; k++)
                if(priv[k] && priv[k][p] < cur) cur = priv[k][p];
            keys[p] = cur;
        }
    }
    for(int k = 0; k < nthreads; k++) free(priv[k]);
    free(priv);
    return ok;
}

void glp_keys_to_framebuffer(const uint64_t* keys, glp_framebuffer_t* fb)
{
    glp_clear(fb);
    const size_t n = (size_t)fb->width * fb->height;
    for(size_t p = 0; p < n; p++)
    {
        const uint32_t q = (uint32_t)(keys[p] >> GLP_KEY_Q_SHIFT);
        if(q >= GLP_Z24_MAX) continue;
        fb->z24[p] = q;
        fb->rgb[3*p+0] = (uint8_t)(keys[p] & 0xFF); fb->rgb[3*p+1] = 0; fb->rgb[3*p+2] = 0;
    }
}
