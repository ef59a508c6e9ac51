/* horizonator_oracle.c -- TEST INFRASTRUCTURE (oracle); see horizonator_oracle.h.
 *
 * Floating-point types follow the reference expression by expression (float where the
 * reference computes in float, double where C promotion makes it double).  Build with
 * -ffp-contract=off.
 */
#define _GNU_SOURCE
#include "horizonator_oracle.h"
#include "gl_pipeline.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define MAXT 4 /* dem.h:8 */

struct oracle_context
{
    /* DEM state, dem.h:10-29 */
    uint8_t* tile[MAXT][MAXT];          /* [i_lon][j_lat], NULL = reads as 0 */
    int origin_lon_lat[2], origin_cellij[2], Ntiles[2];
    int R, cpd;

    /* render state: the uniforms of vertex.glsl */
    glp_uniforms_t u;
    float viewer_lat, viewer_lon;
    int W, H;
    int nthreads;

    int16_t* vertices;                  /* horizonator-lib.c:435-480: (i,j,z) per vertex */
    glp_framebuffer_t fb;
};

/* dem.c:22-76 (no "~/" handling: tests always pass real directories) */
static void tile_path(char* path, size_t n, int lat, int lon, const char* dir)
{
    char ns = lat >= 0 ? 'N' : 'S', we = lon >= 0 ? 'E' : 'W';
    snprintf(path, n, "%s/%c%.2d%c%.3d.hgt", dir, ns, abs(lat), we, abs(lon));
}

/* dem.c:78-243 */
static bool dem_load(oracle_context_t* c, float viewer_lat, float viewer_lon,
                     int radius_cells, float radius_m, const char* dir, bool SRTM1)
{
    if(radius_cells < 0 && radius_m < 0) return false;              /* :90-94 */
    if(radius_cells > 0 && radius_m > 0) return false;              /* :95-99 */

    c->cpd = SRTM1 ? 3600 : 1200;                                   /* :101-104 */
    if(radius_cells > 0)
        c->R = radius_cells;
    else
    {
        const double Rearth = 6371000.0;                            /* :124-126 */
        const double coslat = cos(M_PI / 180.0 * viewer_lat);
        c->R = (int)(0.5 + (double)radius_m / (Rearth * M_PI / 180. * coslat / (double)c->cpd));
    }

    const long expected = (long)(c->cpd + 1) * (c->cpd + 1) * 2;    /* :129-132 */
    const float viewer_lon_lat[2] = { viewer_lon, viewer_lat };

    for(int a = 0; a < 2; a++)                                      /* :136-179 */
    {
        int   icell_origin   = floorf(viewer_lon_lat[a] * c->cpd) - (c->R - 1);
        float origin_lon_lat = (float)icell_origin / (float)c->cpd;
        c->origin_lon_lat[a] = (int)floorf(origin_lon_lat);
        c->origin_cellij[a]  = (int)roundf((origin_lon_lat - c->origin_lon_lat[a]) * c->cpd);

        int last  = c->origin_cellij[a] + c->R * 2 - 1;
        int ilast = last / c->cpd;
        c->Ntiles[a] = ilast + 1;
        if(last == ilast * c->cpd) c->Ntiles[a]--;
        if(c->Ntiles[a] > MAXT) return false;
    }

    for(int j = 0; j < c->Ntiles[1]; j++)                           /* :183-240 */
        for(int i = 0; i < c->Ntiles[0]; i++)
        {
            char path[1024];
            tile_path(path, sizeof(path), j + c->origin_lon_lat[1], i + c->origin_lon_lat[0], dir);
            FILE* f = fopen(path, "rb");
            if(!f) continue;                                        /* missing => 0 */
            fseek(f, 0, SEEK_END);
            long sz = ftell(f);
            fseek(f, 0, SEEK_SET);
            if(sz == 0) { fclose(f); continue; }                    /* empty => 0   */
            if(sz != expected) { fclose(f); return false; }         /* :234-239     */
            c->tile[i][j] = (uint8_t*)malloc(sz);
            if(!c->tile[i][j] || fread(c->tile[i][j], 1, sz, f) != (size_t)sz)
            { fclose(f); return false; }
            fclose(f);
        }
    return true;
}

/* dem.c:264-309 */
int16_t oracle_dem_sample(const oracle_context_t* c, int i, int j)
{
    if(i < 0 || j < 0) return -1;
    int cell[2] = { i + c->origin_cellij[0], j + c->origin_cellij[1] };
    int t[2];
    for(int a = 0; a < 2; a++)
    {
        t[a]     = cell[a] / c->cpd;
        cell[a] -= t[a] * c->cpd;
        if(cell[a] == 0) { t[a]--; cell[a] = c->cpd; }              /* :287-291 */
        if(t[a] >= c->Ntiles[a]) return -1;
        if(t[a] < 0) { t[a] = 0; cell[a] = 0; }  /* reference reads out of bounds here (UB);
                                                    defined as cell 0 of tile 0 */
    }
    const uint8_t* d = c->tile[t[0]][t[1]];
    if(!d) return 0;
    uint32_t p = cell[0] + (c->cpd - cell[1]) * (c->cpd + 1);       /* :300-304 */
    int16_t z = (int16_t)((d[2*p] << 8) | d[2*p + 1]);              /* :307     */
    return z < 0 ? 0 : z;                                           /* :308     */
}

/* horizonator-lib.c:691-816, untextured */
bool oracle_move(oracle_context_t* c, float* viewer_z, float lat, float lon)
{
    float vci = (lon - c->origin_lon_lat[0]) * c->cpd - c->origin_cellij[0];   /* :765-770 */
    float vcj = (lat - c->origin_lon_lat[1]) * c->cpd - c->origin_cellij[1];

    int i0 = (int)floorf(vci), j0 = (int)floorf(vcj);
    float z;
    if(viewer_z == NULL || *viewer_z < 0)                                       /* :778-789 */
    {
        z = fmaxf(fmaxf(oracle_dem_sample(c, i0, j0),     oracle_dem_sample(c, i0 + 1, j0)),
                  fmaxf(oracle_dem_sample(c, i0, j0 + 1), oracle_dem_sample(c, i0 + 1, j0 + 1))) + 1.0;
        if(viewer_z) *viewer_z = z;
    }
    else
        z = *viewer_z;

    c->u.viewer_cell_i  = vci;
    c->u.viewer_cell_j  = vcj;
    c->u.viewer_z       = z;
    c->u.cos_viewer_lat = cosf(lat * M_PI / 180.0f);                            /* :799 */
    c->viewer_lat = lat;
    c->viewer_lon = lon;
    return true;
}

/* horizonator-lib.c:818-836: stored as given */
bool oracle_pan_zoom(oracle_context_t* c, float az_deg0, float az_deg1)
{
    c->u.az_deg0 = az_deg0;
    c->u.az_deg1 = az_deg1;
    return true;
}

/* horizonator-lib.c:864-885 */
bool oracle_set_zextents(oracle_context_t* c, float znear, float zfar, float znc, float zfc)
{
    if(!(znear > 0.0f && znc > 0.0f && zfar > 0.0f && zfc > 0.0f)) return false;
    c->u.znear = znear; c->u.zfar = zfar; c->u.znear_color = znc; c->u.zfar_color = zfc;
    return true;
}

oracle_context_t* oracle_init(float lat, float lon, float* viewer_z, int W, int H,
                              int radius_cells, float radius_m, bool SRTM1, const char* dir)
{
    oracle_context_t* c = (oracle_context_t*)calloc(1, sizeof(*c));
    if(!c) return NULL;
    c->nthreads = 1;
    if(!dem_load(c, lat, lon, radius_cells, radius_m, dir, SRTM1)) { oracle_deinit(c); return NULL; }

    /* horizonator-lib.c:435-480: j (north) outer, i (east) inner */
    const int N = 2 * c->R;
    c->vertices = (int16_t*)malloc((size_t)N * N * 3 * sizeof(int16_t));
    if(!c->vertices) { oracle_deinit(c); return NULL; }
    size_t k = 0;
    for(int j = 0; j < N; j++)
        for(int i = 0; i < N; i++)
        {
            c->vertices[k++] = (int16_t)i;
            c->vertices[k++] = (int16_t)j;
            c->vertices[k++] = oracle_dem_sample(c, i, j);
        }

    c->u.DEG_PER_CELL = 1.0f / (float)c->cpd;                       /* :577 */
    oracle_move(c, viewer_z, lat, lon);                             /* :611 */
    oracle_set_zextents(c, 100.0f, 40000.0f, 100.0f, 40000.0f);     /* :612-614 */

    c->W = W; c->H = H;
    c->u.aspect = (float)W / (float)H;                              /* :658-659 */
    if(!glp_framebuffer_alloc(&c->fb, W, H)) { oracle_deinit(c); return NULL; }
    oracle_pan_zoom(c, -45.f, 45.f);                                /* :670 */
    return c;
}

void oracle_deinit(oracle_context_t* c)
{
    if(!c) return;
    for(int i = 0; i < MAXT; i++) for(int j = 0; j < MAXT; j++) free(c->tile[i][j]);
    free(c->vertices);
    glp_framebuffer_free(&c->fb);
    free(c);
}

void oracle_set_threads(oracle_context_t* c, int n) { c->nthreads = n < 1 ? 1 : n; }

void oracle_get_dem_geometry(const oracle_context_t* c, int out[8])
{
    out[0] = c->origin_lon_lat[0]; out[1] = c->origin_lon_lat[1];
    out[2] = c->origin_cellij[0];  out[3] = c->origin_cellij[1];
    out[4] = c->Ntiles[0];         out[5] = c->Ntiles[1];
    out[6] = c->R;                 out[7] = c->cpd;
}
void oracle_get_viewer(const oracle_context_t* c, float o[4])
{
    o[0] = c->u.viewer_cell_i; o[1] = c->u.viewer_cell_j; o[2] = c->u.viewer_z; o[3] = c->u.cos_viewer_lat;
}

/* horizonator-lib.c:936-1048: image and ranges out of the framebuffer, top row first */
static void read_back(const glp_framebuffer_t* fb, const glp_uniforms_t* u, char* image, float* ranges)
{
    const int W = fb->width, H = fb->height;
    if(image)                                                       /* :936-959 */
    {
        uint8_t* tmp = (uint8_t*)malloc((size_t)W * H * 3);
        glp_read_bgr(fb, tmp);
        for(int y = 0; y < H; y++)   /* GL row y -> image row H-1-y */
            memcpy(image + (size_t)(H - 1 - y) * W * 3, tmp + (size_t)y * W * 3, (size_t)W * 3);
        free(tmp);
    }
    if(ranges)                                                      /* :960-1048 */
    {
        float* depth = (float*)malloc((size_t)W * H * sizeof(float));
        glp_read_depth_float(fb, 0, 0, W, H, depth);

        const float az_deg0 = u->az_deg0, az_deg1 = u->az_deg1;
        const float znear = u->znear, zfar = u->zfar;
        const float aspect = (float)W / (float)H;                   /* :1006 */

        for(int y = 0; y < H; y++)   /* y = GL row */
        {
            /* :1007-1012 evaluates tan(el) for rows of the lower half and negates it for
               the mirrored row; the centre row of an odd height is evaluated directly */
            int   ysrc = (y < H / 2 || ((H & 1) && y == H / 2)) ? y : H - 1 - y;
            float el_ndc = ((float)ysrc + 0.5f) / (float)H * 2.f - 1.f;
            float el     = el_ndc * (az_deg1 - az_deg0) / 2.f / aspect * M_PI / 180.0f;
            float tanel  = tanf(el);
            if(ysrc != y) tanel = -tanel;

            for(int x = 0; x < W; x++)
            {
                float d = depth[(size_t)y * W + x], out;
                if(d == 1.0f) out = -1.0f;                          /* :1016 */
                else
                {
                    float length_en = d * (zfar - znear) + znear;   /* :1018 */
                    float z = tanel * length_en;
                    out = hypotf(length_en, z);                     /* :1023-1024 */
                }
                ranges[(size_t)(H - 1 - y) * W + x] = out;
            }
        }
        free(depth);
    }
}

/* horizonator-lib.c:911-1051 */
bool oracle_render_offscreen(oracle_context_t* c, char* image, float* ranges)
{
    const int N = 2 * c->R;

    /* :887-899 redraw: clear, then every triangle of the dense grid in index order */
    glp_clear(&c->fb);
    glp_draw_triangles(&c->fb, &c->u, c->vertices, (int64_t)N * N,
                       NULL, (int64_t)2 * (N - 1) * (N - 1), N, c->nthreads);
    read_back(&c->fb, &c->u, image, ranges);
    return true;
}

float oracle_vertex_stage(const oracle_context_t* c, glp_vtx_t* out)
{
    const int N = 2 * c->R;
    glp_vertices(&c->u, c->vertices, (int64_t)N * N, c->W, c->H, out, c->nthreads);
    return glp_seam_period(&c->u);
}

bool oracle_read_keys(const uint64_t* keys, int W, int H, float az_deg0, float az_deg1, float znear, float zfar,
                      char* image, float* ranges)
{
    glp_framebuffer_t fb;
    if(!glp_framebuffer_alloc(&fb, W, H)) return false;
    glp_uniforms_t u;
    memset(&u, 0, sizeof(u));
    u.az_deg0 = az_deg0; u.az_deg1 = az_deg1; u.znear = znear; u.zfar = zfar;
    glp_keys_to_framebuffer(keys, &fb);
    read_back(&fb, &u, image, ranges);
    glp_framebuffer_free(&fb);
    return true;
}

void oracle_set_curvature(oracle_context_t* c, float coefficient) { c->u.curvature = coefficient; }
void oracle_set_seam_wrap(oracle_context_t* c, bool on) { c->u.seam_wrap = on ? 1 : 0; }
