/* viewshed_oracle.c -- TEST INFRASTRUCTURE (oracle).  Not part of the product; only tests/ and tools may use it.
 *
 * Viewsheds of an oracle context's current eye (oracle_move) over the N x N vertices of its DEM square (N = 2R),
 * not in the reference:
 *   vs_oracle_r2     R2 ray casting exactly as include/horizonator-batch.h defines it, operation for operation in
 *                    float -- the GPU kernel (k_viewshed) must match it bit for bit
 *   vs_oracle_exact  brute-force line of sight on the reference's triangulation, in double (small scenes only)
 * Heights come from vs_oracle_mosaic() (oracle_dem_sample, dem.c:264-309), the eye from oracle_get_viewer(), the cell
 * size from oracle_get_dem_geometry(): only the public interface of horizonator_oracle.h.
 * mask: N x W32 uint32, W32 = (N + 31) / 32, cell i of row j = bit (i & 31) of word [j][i >> 5]; overwritten.
 * Both return false (mask untouched) when the eye is not inside [0, N-1)^2.
 *
 * Build with -ffp-contract=off, like the rest of oracle/: one IEEE rounding per source operator.
 */
#include "horizonator_oracle.h"

#include <math.h>
#include <stdbool.h>
#include <stdint.h>
#include <string.h>

typedef struct
{
    const int16_t* z;                   /* [N][N], row j north, column i east */
    int N, w32;
    float vci, vcj, vz, cosl, dpc, curv;
} vs_scene_t;

static const float vs_Rearth = 6371000.0f;          /* vertex.glsl:30 */
static const float vs_pi     = 3.14159265358979f;   /* vertex.glsl:31 */

/* the square's heights, N x N int16 */
void vs_oracle_mosaic(const oracle_context_t* ctx, int16_t* out)
{
    int g[8];
    oracle_get_dem_geometry(ctx, g);
    const int N = 2 * g[6];
    #pragma omp parallel for schedule(static)
    for(int j = 0; j < N; j++)
        for(int i = 0; i < N; i++) out[(size_t)j * N + i] = oracle_dem_sample(ctx, i, j);
}

static bool vs_scene(const oracle_context_t* ctx, const int16_t* z, float curvature, vs_scene_t* s)
{
    int g[8];
    float v[4];
    oracle_get_dem_geometry(ctx, g);
    oracle_get_viewer(ctx, v);
    s->z = z; s->N = 2 * g[6]; s->w32 = (s->N + 31) / 32;
    s->vci = v[0]; s->vcj = v[1]; s->vz = v[2]; s->cosl = v[3];
    s->dpc = 1.0f / (float)g[7];                                    /* horizonator-lib.c:577 */
    s->curv = curvature;
    const float N1 = (float)(s->N - 1);
    return s->vci >= 0.f && s->vci < N1 && s->vcj >= 0.f && s->vcj < N1;
}

static float vs_height(const vs_scene_t* s, int i, int j) { return (float)s->z[(size_t)j * s->N + i]; }

/* metres from the eye along one axis at cell coordinate x: vertex.glsl:128-130 with x in place of the vertex
   index; scale = cos_viewer_lat east, 1 north (x * 1.0f == x) */
static float vs_metres(float x, float v, float dpc, float scale)
{
    return (x - v) * dpc * vs_Rearth * vs_pi / 180.f * scale;
}

static void vs_set(uint32_t* mask, int w32, int i, int j)
{
    uint32_t* w = mask + (size_t)j * w32 + (i >> 5);
    const uint32_t bit = 1u << (i & 31);
    #pragma omp atomic
    *w |= bit;
}

/* the four vertices around the eye */
static void vs_eye_cell(const vs_scene_t* s, uint32_t* mask)
{
    const int i0 = (int)floorf(s->vci), j0 = (int)floorf(s->vcj);
    for(int dj = 0; dj < 2; dj++)
        for(int di = 0; di < 2; di++) vs_set(mask, s->w32, i0 + di, j0 + dj);
}

/* boundary vertex k of 4N-4: the bottom row, the top row, then the left and the right column without corners */
static void vs_target(int N, int k, int* ti, int* tj)
{
    if(k < N)              { *ti = k;     *tj = 0;     }
    else if(k < 2 * N)     { *ti = k - N; *tj = N - 1; }
    else if(k < 3 * N - 2) { *ti = 0;     *tj = k - 2 * N + 1; }
    else                   { *ti = N - 1; *tj = k - (3 * N - 2) + 1; }
}

/* One ray of R2 (horizonator-batch.h): "a" is the axis it steps along, "b" the other one. */
static void vs_ray(const vs_scene_t* s, float th, int ti, int tj, uint32_t* mask)
{
    const int N = s->N;
    const float vci = s->vci, vcj = s->vcj, vz = s->vz, dpc = s->dpc, curv = s->curv;
    const float di = (float)ti - vci, dj = (float)tj - vcj;
    const bool xmaj = fabsf(di) >= fabsf(dj);
    const float va = xmaj ? vci : vcj, vb = xmaj ? vcj : vci;
    const float da = xmaj ? di : dj, db = xmaj ? dj : di;
    const float sa = xmaj ? s->cosl : 1.0f, sb = xmaj ? 1.0f : s->cosl;
    const int ta = xmaj ? ti : tj;
    if(da == 0.f) return;                                   /* the eye sits on this boundary vertex */
    const float slope = db / da;
    const int step = da > 0.f ? 1 : -1;
    const int a0 = da > 0.f ? (int)floorf(va) + 1 : (int)ceilf(va) - 1;
    float smax = -INFINITY;
    for(int a = a0;; a += step)
    {
        const float b = vb + ((float)a - va) * slope;
        int b0 = (int)floorf(b);
        b0 = b0 < 0 ? 0 : (b0 > N - 2 ? N - 2 : b0);
        int r = (int)rintf(b);
        r = r < 0 ? 0 : (r > N - 1 ? N - 1 : r);
        const float z0 = xmaj ? vs_height(s, a, b0) : vs_height(s, b0, a);
        const float z1 = xmaj ? vs_height(s, a, b0 + 1) : vs_height(s, b0 + 1, a);
        /* the surface at (a, b): linear along the grid edge between b0 and b0 + 1 */
        const float t = b - (float)b0;
        const float z = z0 + (z1 - z0) * t;
        const float ma = vs_metres((float)a, va, dpc, sa), mb = vs_metres(b, vb, dpc, sb);
        const float d2 = ma * ma + mb * mb;
        const float sl = (z - vz - curv * d2) / sqrtf(d2);
        /* the vertex this step decides: (a, rint(b)) against the steps before it */
        const float zr = r == b0 ? z0 : z1;
        const float mr = vs_metres((float)r, vb, dpc, sb);
        const float d2r = ma * ma + mr * mr;
        const float q = (zr - vz - curv * d2r + th) / sqrtf(d2r);
        if(q >= smax) vs_set(mask, s->w32, xmaj ? a : r, xmaj ? r : a);
        smax = sl > smax ? sl : smax;
        if(a == ta) break;
    }
}

bool vs_oracle_r2(const oracle_context_t* ctx, const int16_t* z, float curvature, float target_height, int nthreads,
                  uint32_t* mask)
{
    vs_scene_t s;
    if(!vs_scene(ctx, z, curvature, &s)) return false;
    const int N = s.N;
    memset(mask, 0, (size_t)N * s.w32 * sizeof(uint32_t));
    vs_eye_cell(&s, mask);
    #pragma omp parallel for num_threads(nthreads < 1 ? 1 : nthreads) schedule(dynamic, 64)
    for(int k = 0; k < 4 * N - 4; k++)
    {
        int ti, tj;
        vs_target(N, k, &ti, &tj);
        vs_ray(&s, target_height, ti, tj, mask);
    }
    return true;
}

/* height of the triangulated surface (horizonator-lib.c:496-508: the cell (i,j) is split along its (i,j)-(i+1,j+1)
   diagonal) at a vertex, double precision */
static double vs_zd(const vs_scene_t* s, int i, int j) { return (double)s->z[(size_t)j * s->N + i]; }

bool vs_oracle_exact(const oracle_context_t* ctx, const int16_t* z, float curvature, float target_height, int nthreads,
                     uint32_t* mask)
{
    vs_scene_t s;
    if(!vs_scene(ctx, z, curvature, &s)) return false;
    const int N = s.N;
    memset(mask, 0, (size_t)N * s.w32 * sizeof(uint32_t));
    vs_eye_cell(&s, mask);
    const double vci = s.vci, vcj = s.vcj, vz = s.vz, curv = s.curv;
    const double cn = (double)s.dpc * 6371000.0 * M_PI / 180.0, ce = cn * (double)s.cosl;
    const int ei = (int)floorf(s.vci), ej = (int)floorf(s.vcj);
    #pragma omp parallel for num_threads(nthreads < 1 ? 1 : nthreads) schedule(dynamic, 1)
    for(int tj = 0; tj < N; tj++)
        for(int ti = 0; ti < N; ti++)
        {
            if((ti == ei || ti == ei + 1) && (tj == ej || tj == ej + 1)) continue;
            const double Di = ti - vci, Dj = tj - vcj;
            const double dT = sqrt(Di * ce * Di * ce + Dj * cn * Dj * cn);
            const double sT = (vs_zd(&s, ti, tj) - vz - curv * dT * dT + target_height) / dT;
            /* the segment's horizontal projection crosses vertical lines i = k, horizontal lines j = k and diagonals
               i - j = k; between crossings the surface under it is linear, so the crossings decide */
            bool vis = true;
            for(int kind = 0; kind < 3 && vis; kind++)
            {
                const double p0 = kind == 0 ? vci : kind == 1 ? vcj : vci - vcj;
                const double dp = kind == 0 ? Di : kind == 1 ? Dj : Di - Dj;
                if(dp == 0.0) continue;
                const double lo = fmin(p0, p0 + dp), hi = fmax(p0, p0 + dp);
                for(int k = (int)ceil(lo); k <= (int)floor(hi) && vis; k++)
                {
                    const double t = ((double)k - p0) / dp;
                    if(t <= 1e-9 || t >= 1.0 - 1e-9) continue;
                    const double x = vci + t * Di, y = vcj + t * Dj;
                    double zc;
                    if(kind == 0)
                    {
                        int y0 = (int)floor(y); y0 = y0 > N - 2 ? N - 2 : (y0 < 0 ? 0 : y0);
                        zc = vs_zd(&s, k, y0) + (vs_zd(&s, k, y0 + 1) - vs_zd(&s, k, y0)) * (y - y0);
                    }
                    else if(kind == 1)
                    {
                        int x0 = (int)floor(x); x0 = x0 > N - 2 ? N - 2 : (x0 < 0 ? 0 : x0);
                        zc = vs_zd(&s, x0, k) + (vs_zd(&s, x0 + 1, k) - vs_zd(&s, x0, k)) * (x - x0);
                    }
                    else
                    {
                        int x0 = (int)floor(x); x0 = x0 > N - 2 ? N - 2 : (x0 < 0 ? 0 : x0);
                        const int y0 = x0 - k;
                        if(y0 < 0 || y0 > N - 2) continue;
                        zc = vs_zd(&s, x0, y0) + (vs_zd(&s, x0 + 1, y0 + 1) - vs_zd(&s, x0, y0)) * (x - x0);
                    }
                    const double d = t * dT;
                    if((zc - vz - curv * d * d) / d > sT) vis = false;
                }
            }
            if(vis) vs_set(mask, s.w32, ti, tj);
        }
    return true;
}
