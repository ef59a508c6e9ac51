// hz_kernels.cu -- sm_100a kernels of libhorizonator's render path.
//
//   k_mosaic   (init)    raw big-endian .hgt tiles -> one int16 mosaic        replaces dem.c:264-309 called
//                                                                              (2R)^2 times at horizonator-lib.c:435-439
//   k_minmax_* (init)    (min,max) height per 4x4-cell block and per 32x32-cell tile: the culling pyramid
//   k_prepare  (render)  clear visibility keys, per-column/row metre tables    glClear, lib:896; vertex.glsl:128-130
//   k_near     (render)  the tiles around the eye: mesh generation, projection,  lib:496-508 (index pattern), vertex.glsl,
//                        exact integer cull -> list of triangles                  GL cull/clip
//   k_tiles, k_blocks / k_blocks_mid, k_mesh (render)
//                        the rest of the mesh in bands outwards from the eye: whole tiles, then blocks (for the views
//                        of a batch with 8x8-cell squares in between: k_blocks_mid), are dropped by conservative tests
//                        (beyond zfar, no pixel centre of the target inside their screen box, everything in that box
//                        already nearer in the visibility buffer); what is left goes through the same exact stages
//                        as in k_near -> list of triangles
//   k_raster   (render)  set-up, rasterisation and depth test of a list,          vertex.glsl, geometry.glsl, GL raster,
//                        one thread per triangle                                  depth test, fragment.glsl
//   k_big      (render)  the triangles with large bounding boxes, one warp per 32-column sub-box (lane = column)
//   k_peer_barrier (multi-GPU)  barrier between the ranks of a wedge-sharded panorama through peer memory
//   k_resolve4 / k_resolve1 (render)  keys -> BGR8 image + float range image, top row first   lib:936-1048
//   k_horizon  (extra)   range image -> per-column topmost terrain row and its range
//   k_viewshed, k_viewshed_count (viewsheds)  R2 ray casting over the DEM square, one thread per ray -> bit masks;
//                        masks -> per-vertex counts of the views that see it
//
// The mesh is never materialised: triangle t of the reference's index buffer is (cell = t>>1, half = t&1)
// and its vertices are read straight from the int16 mosaic.
//
// Compiled with -fmad=false: plain a*b+c is two IEEE roundings (see hz_math.cuh).
#include "hz_device.h"
#include "hz_math.cuh"

#include <cstdint>
#include <cstdlib>

// ---- launches ----------------------------------------------------------------------------------
// A render is a chain of a dozen short kernels on one stream.  Each is launched with programmatic stream
// serialisation (PDL): its CTAs may be placed on the SMs while the previous kernel is still draining, and wait at
// hz_wait_for_previous_kernel() -- part of the prologue of every render kernel -- until that kernel has completed
// and its writes are visible.  That hides most of the launch latency between the kernels; the ordering is unchanged.
__device__ __forceinline__ void hz_wait_for_previous_kernel()
{
    cudaGridDependencySynchronize();
    cudaTriggerProgrammaticLaunchCompletion();
}

// First statements of every render kernel: the CTA copies its parameter block (written by the host->device copy
// that precedes the whole chain, not by an earlier kernel of it) into shared memory BEFORE it waits for the previous
// kernel, so that those reads overlap that kernel's tail instead of following it; afterwards every P.field is a
// shared-memory read.
// One launch serves gridDim.y views: view y reads its copy of the launch's variant, HZ_V_COUNT elements per view on.
// (Every render kernel runs CTAs of HZ_CTA_THREADS threads and the block has fewer 16-byte units than that: one guarded
// 128-bit load per thread.  Written as a loop striding by blockDim.x the compiler does not know the trip count and
// works it out with an integer division -- some 50 instructions at the head of every warp of every launch.)
#define HZ_CTA_THREADS 256
static_assert(sizeof(HzView) % 16 == 0 && sizeof(HzView) / 16 <= HZ_CTA_THREADS && alignof(HzView) == 16, "HzView: whole 16-byte units");
#define HZ_KERNEL_PROLOGUE(V, P)                                                                           \
    __shared__ HzView hz_s_view;                                                                           \
    if(threadIdx.x < sizeof(HzView) / 16)                                                                  \
        ((uint4*)&hz_s_view)[threadIdx.x] = __ldg((const uint4*)((V) + blockIdx.y * HZ_V_COUNT) + threadIdx.x); \
    __syncthreads();                                                                                       \
    hz_wait_for_previous_kernel();                                                                         \
    const HzView& P = hz_s_view

// The kernels whose amount of work is only known on the device (queue lengths) are launched with a multiple of the SM
// count and loop: ctas_per_sm as tuned for a lone view, times v.grid_percent/100.  Views that render concurrently
// (the lanes of a batch) do better with smaller grids -- most CTAs of a worst-case grid find nothing to do, and
// their launch and prologue compete with the other views' real work -- a lone view with larger ones.
// With several views per launch (gridDim.y) that total is divided among them.
static unsigned int hz_grid(const HzView& v, unsigned int ctas_per_sm, int nviews)
{
    const unsigned int nv = (unsigned int)(nviews > 0 ? nviews : 1);
    const unsigned int total = 148u * ctas_per_sm * (unsigned int)(v.grid_percent > 0 ? v.grid_percent : 100) / 100u;
    const unsigned int g = (total + nv - 1u) / nv, floor_ = 148u / nv > 8u ? 148u / nv : 8u;
    return g < floor_ ? floor_ : g;
}

template <typename... KArgs, typename... Args>
static cudaError_t hz_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, Args&&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ================================================================================================
// k_mosaic
// ================================================================================================

// dem.c:278-293 for one axis: mosaic index -> (tile, cell inside tile).  Cell 0 of a tile is read from the
// previous tile's last row/column (tiles overlap by one sample); with no previous tile the reference reads
// out of bounds, here it reads cell 0 of tile 0.
__device__ __forceinline__ void hz_split_cell(int g, int cpd, int& t, int& c)
{
    t = g / cpd;
    c = g - t * cpd;
    if(c == 0) { t--; c = cpd; }
    if(t < 0)  { t = 0; c = 0; }
}

__device__ __forceinline__ int16_t hz_decode_be16(const uint8_t* p)
{
    const int16_t z = (int16_t)(((unsigned)p[0] << 8) | (unsigned)p[1]);   // dem.c:307
    return z < 0 ? (int16_t)0 : z;                                          // dem.c:308
}

// Each thread produces 8 consecutive samples of one mosaic row (one 16-byte store).  When the 8 samples come
// from one tile row they are fetched with aligned 32-bit loads, byte-swapped with PRMT and clamped two at a
// time; otherwise (tile boundary) sample by sample.
__global__ void __launch_bounds__(128)
k_mosaic(const HzTiles T, int16_t* __restrict__ out, int N, int pitch)
{
    const int j  = blockIdx.y;
    const int i0 = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
    if(i0 >= pitch) return;

    const int cpd = T.cpd;
    int tj, cj;
    hz_split_cell(j + T.origin_cell[1], cpd, tj, cj);
    const size_t row_off = (size_t)(cpd - cj) * (size_t)(cpd + 1);          // dem.c:300-304: north row first

    uint32_t w[4] = {0, 0, 0, 0};    // 8 little-endian int16, clamped

    int ti0, ci0;
    hz_split_cell(i0 + T.origin_cell[0], cpd, ti0, ci0);
    const bool one_run = (i0 + 8 <= N) && (ci0 >= 1) && (ci0 + 7 <= cpd) && (tj < T.ntiles[1]) && (ti0 < T.ntiles[0]);

    if(one_run)
    {
        const uint8_t* tile = T.tile[ti0][tj];
        if(tile != nullptr)
        {
            const uint8_t* src = tile + 2 * (row_off + (size_t)ci0);
            const uintptr_t a  = (uintptr_t)src;
            const uint32_t* s4 = (const uint32_t*)(a & ~(uintptr_t)3);
            uint32_t r[5];
            #pragma unroll
            for(int k = 0; k < 4; k++) r[k] = __ldg(s4 + k);
            if(a & 2)
            {
                r[4] = __ldg(s4 + 4);
                #pragma unroll
                for(int k = 0; k < 4; k++) r[k] = __funnelshift_r(r[k], r[k + 1], 16);
            }
            #pragma unroll
            for(int k = 0; k < 4; k++)
            {
                const uint32_t sw = __byte_perm(r[k], 0, 0x2301);           // swap bytes inside each half
                w[k] = __vmaxs2(sw, 0u);                                     // per-half max(z, 0)
            }
        }
    }
    else
    {
        #pragma unroll
        for(int k = 0; k < 8; k++)
        {
            const int i = i0 + k;
            int16_t z = 0;
            if(i < N)
            {
                int ti, ci;
                hz_split_cell(i + T.origin_cell[0], cpd, ti, ci);
                if(ti >= T.ntiles[0] || tj >= T.ntiles[1]) z = -1;          // dem.c:293
                else
                {
                    const uint8_t* tile = T.tile[ti][tj];
                    if(tile != nullptr) z = hz_decode_be16(tile + 2 * (row_off + (size_t)ci));
                }
            }
            w[k >> 1] |= (uint32_t)(uint16_t)z << (16 * (k & 1));
        }
    }
    *(uint4*)(out + (size_t)j * pitch + i0) = make_uint4(w[0], w[1], w[2], w[3]);
}

cudaError_t hz_launch_mosaic(const HzTiles& t, int16_t* mosaic, int N, int pitch, cudaStream_t stream)
{
    dim3 block(128), grid((pitch / 8 + 127) / 128, N);
    k_mosaic<<<grid, block, 0, stream>>>(t, mosaic, N, pitch);
    return cudaGetLastError();
}

// ================================================================================================
// k_prepare
// ================================================================================================

__global__ void __launch_bounds__(256)
k_prepare(const HzView* __restrict__ V)
{
    HZ_KERNEL_PROLOGUE(V, P);
    const unsigned int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned int nth = gridDim.x * blockDim.x;

    // glClear: depth 1.0 everywhere -- only when the epoch of the keys has wrapped (see the visibility key): then the
    // whole buffer is cleared, two keys at a time (16-byte stores), four stores per trip
    const size_t nkeys = P.clear_keys;
    if(nkeys)
    {
        const unsigned int npairs = (unsigned int)(nkeys / 2);
        ulonglong2* v2 = (ulonglong2*)P.vis;
        const ulonglong2 clear2 = make_ulonglong2(HZ_KEY_CLEAR, HZ_KEY_CLEAR);
        unsigned int k = tid;
        for(; k + 3u * nth < npairs; k += 4u * nth)
        {
            v2[k] = clear2; v2[k + nth] = clear2; v2[k + 2u * nth] = clear2; v2[k + 3u * nth] = clear2;
        }
        for(; k < npairs; k += nth) v2[k] = clear2;
        if(tid == 0 && (nkeys & 1)) P.vis[nkeys - 1] = HZ_KEY_CLEAR;
    }

    // vertex.glsl:128-130, operator by operator:
    //   e = (i - viewer_cell_i) * DEG_PER_CELL * Rearth * pi/180. * cos_viewer_lat
    //   n = (j - viewer_cell_j) * DEG_PER_CELL * Rearth * pi/180.
    // (HZ_MESH_PAD more than the mesh has: the last blocks may hang over its edge, see hz_group_vertex)
    for(unsigned int c = tid; c < (unsigned int)(P.N + HZ_MESH_PAD); c += nth)
    {
        const float f = (float)(int)c;
        P.e_tab[c] = (f - P.viewer_cell_i) * P.deg_per_cell * HZ_REARTH_F * HZ_PI_F / 180.f * P.cos_viewer_lat;
        P.n_tab[c] = (f - P.viewer_cell_j) * P.deg_per_cell * HZ_REARTH_F * HZ_PI_F / 180.f;
    }
    if(tid < (unsigned int)P.ncounters) P.counters[tid] = 0;
}

cudaError_t hz_launch_prepare(const HzView& v, const HzView* d_v, int nviews, cudaStream_t stream)
{
    // enough threads to keep the stores of the clear flowing; the axis tables take a few trips
    unsigned int blocks = 148u * 2u;
    if(nviews > 1) blocks = 148u * 8u / (unsigned int)nviews;
    if(blocks < 16u) blocks = 16u;
    (void)v;
    return hz_launch(k_prepare, dim3(blocks, (unsigned)nviews), dim3(256), stream, d_v);
}

// ================================================================================================
// projection and triangle set-up shared by the mesh kernels, k_raster and k_big
// ================================================================================================

#define HZ_GUARD_PX   2097152.0f      /* 2^21: triangles reaching beyond are dropped (oracle rule F5) */
#define HZ_SNAP_LIMIT 536870912.0f    /* 2^29 = guard band in 1/256 pixel */

struct HzVtx
{
    float xn, yn;    // gl_Position.x, gl_Position.y
    float z;         // terrain height, metres
};

// vertex.glsl:132-153 for one vertex at (e, n) metres from the eye with terrain height z
__device__ __forceinline__ void hz_project(const HzView& P, float e, float n, float z, HzVtx& v)
{
    const float d2 = e * e + n * n;
    const float h  = z - P.viewer_z - P.curvature * d2;      // curvature is 0 unless the caller opted in: exactly z - viewer_z
    float az = hz_atan2_az(e, n);
    // unwrap_near_rad(az, az_rad_center), vertex.glsl:34-38; the division by 2*pi is a multiplication by
    // the rounded reciprocal here (the quotient only has to pick the right turn count)
    const float t = (az - P.az_center) * 0.15915494309189535f;
    az = (t - rintf(t)) * 2.f * HZ_PI_F + P.az_center;
    v.xn = (az - P.az_center) * P.az_ndc_per_rad;
    v.yn = hz_atan_el(h, d2) * P.aspect * P.az_ndc_per_rad;
    v.z  = z;
}

// window coordinate -> 1/256 pixel fixed point (oracle rule F2), saturated at the guard band so that the
// integer math downstream cannot overflow (triangles touching the guard band are dropped anyway)
__device__ __forceinline__ int hz_snap(float a)
{
    float t = a * 256.0f;
    if(fabsf(t) < 8388608.0f) t = floorf(t + 0.5f);
    t = fminf(fmaxf(t, -HZ_SNAP_LIMIT), HZ_SNAP_LIMIT);
    return (int)t;
}

#define HZ_ID_LOD_SHIFT 29                     /* see the visibility key in hz_device.h */
#define HZ_ID_CELL_MASK 0x1FFFFFFFu

// triangle number -> its three vertices (row j, column i), lib:496-508; s = 1 unless the triangle belongs to a band
// meshed at a coarser (opt-in) level of detail
__device__ __forceinline__ void hz_tri_vertices(unsigned int id, int N, int vj[3], int vi[3])
{
    const int s = 1 << (id >> HZ_ID_LOD_SHIFT);
    const unsigned int cell = (id & HZ_ID_CELL_MASK) >> 1;
    const int j = (int)(cell / (unsigned int)(N - 1)), i = (int)(cell % (unsigned int)(N - 1));
    vj[0] = j; vi[0] = i;
    if((id & 1u) == 0) { vj[1] = j + s; vi[1] = i + s; vj[2] = j + s; vi[2] = i;     }
    else               { vj[1] = j;     vi[1] = i + s; vj[2] = j + s; vi[2] = i + s; }
}

struct HzTri
{
    int X0, Y0, X1, Y1, X2, Y2;      // snapped window positions, 1/256 pixel
    int px0, px1, py0, py1;          // clipped pixel bounding box (inclusive)
    float xw0, yw0, xw1, yw1, xw2, yw2;
    // attribute planes through the unsnapped float vertices, anchored at vertex 0 (oracle rule F6)
    float z0w, r0, dzdx, dzdy, drdx, drdy;
    float zw_lo, zw_hi;              // F6: the interpolated depth stays within the vertex depths widened 4x
    unsigned int id;
};

enum { HZ_SETUP_NOTHING = 0, HZ_SETUP_OK = 1, HZ_SETUP_TOO_WIDE = -1, HZ_SETUP_QUEUE_FULL = -2 };

// geometry.glsl:21-27, guard band, back-face cull, bounding box.  HZ_SETUP_OK, or why the triangle produces nothing.
__device__ __forceinline__ int
hz_tri_bounds(const HzView& P, const HzVtx& a, const HzVtx& b, const HzVtx& c, HzTri& T)
{
    const float xmax = fmaxf(fmaxf(a.xn, b.xn), c.xn);
    const float xmin = fminf(fminf(a.xn, b.xn), c.xn);
    if(xmax - xmin > 0.5f) return HZ_SETUP_TOO_WIDE;                         // geometry.glsl:21-27

    const float halfW = 0.5f * (float)P.W, halfH = 0.5f * (float)P.H;
    T.xw0 = a.xn * halfW + halfW; T.yw0 = a.yn * halfH + halfH;              // viewport transform (F1)
    T.xw1 = b.xn * halfW + halfW; T.yw1 = b.yn * halfH + halfH;
    T.xw2 = c.xn * halfW + halfW; T.yw2 = c.yn * halfH + halfH;
    if(!(fabsf(T.xw0) < HZ_GUARD_PX && fabsf(T.yw0) < HZ_GUARD_PX &&
         fabsf(T.xw1) < HZ_GUARD_PX && fabsf(T.yw1) < HZ_GUARD_PX &&
         fabsf(T.xw2) < HZ_GUARD_PX && fabsf(T.yw2) < HZ_GUARD_PX)) return HZ_SETUP_NOTHING;   // F5

    T.X0 = hz_snap(T.xw0); T.Y0 = hz_snap(T.yw0);
    T.X1 = hz_snap(T.xw1); T.Y1 = hz_snap(T.yw1);
    T.X2 = hz_snap(T.xw2); T.Y2 = hz_snap(T.yw2);

    // GL_CULL_FACE, front = counter-clockwise, y up (lib:184; F3)
    const long long area = (long long)(T.X1 - T.X0) * (T.Y2 - T.Y0) - (long long)(T.X2 - T.X0) * (T.Y1 - T.Y0);
    if(area <= 0) return HZ_SETUP_NOTHING;

    const int bx0 = min(min(T.X0, T.X1), T.X2), bx1 = max(max(T.X0, T.X1), T.X2);
    const int by0 = min(min(T.Y0, T.Y1), T.Y2), by1 = max(max(T.Y0, T.Y1), T.Y2);
    // pixel centres sit at 256*p + 128
    T.px0 = max((bx0 + 127) >> 8, P.x0);
    T.px1 = min((bx1 - 128) >> 8, P.x1 - 1);
    T.py0 = max((by0 + 127) >> 8, 0);
    T.py1 = min((by1 - 128) >> 8, P.H - 1);
    return (T.px0 <= T.px1 && T.py0 <= T.py1) ? HZ_SETUP_OK : HZ_SETUP_NOTHING;
}

// vertex.glsl:155,159-160 for one vertex: window depth and red channel
__device__ __forceinline__ void hz_depth_shade(const HzView& P, float e, float n, float z, float& zw, float& r)
{
    const float d2  = e * e + n * n;
    const float h   = z - P.viewer_z - P.curvature * d2;
    const float dne = sqrtf(d2);                                             // length(en)
    const float len = sqrtf(d2 + h * h);                                     // length(enh)
    const float zn  = (len - P.znear) / (P.zfar - P.znear) * 2.f - 1.f;
    zw = zn * 0.5f + 0.5f;                                                   // glDepthRange(0,1)
    r  = fmaxf(fminf((dne - P.znear_color) / (P.zfar_color - P.znear_color), 1.0f), 0.0f);
}

__device__ __forceinline__ void
hz_tri_planes(const HzView& P, HzTri& T,
              float e0, float n0, float z0, float e1, float n1, float z1, float e2, float n2, float z2)
{
    float zw0, zw1, zw2, r0, r1, r2;
    hz_depth_shade(P, e0, n0, z0, zw0, r0);
    hz_depth_shade(P, e1, n1, z1, zw1, r1);
    hz_depth_shade(P, e2, n2, z2, zw2, r2);

    const float ax = T.xw1 - T.xw0, ay = T.yw1 - T.yw0;
    const float bx = T.xw2 - T.xw0, by = T.yw2 - T.yw0;
    const float det = ax * by - bx * ay;
    const float inv = 1.0f / det;
    const float az = zw1 - zw0, bz = zw2 - zw0;
    const float ar = r1 - r0,   br = r2 - r0;
    T.dzdx = (az * by - bz * ay) * inv;
    T.dzdy = (bz * ax - az * bx) * inv;
    T.drdx = (ar * by - br * ay) * inv;
    T.drdy = (br * ax - ar * bx) * inv;
    T.z0w = zw0; T.r0 = r0;
    const float zw_min = fminf(fminf(zw0, zw1), zw2), zw_max = fmaxf(fmaxf(zw0, zw1), zw2);
    T.zw_lo = zw_min - 4.0f * (zw_max - zw_min);
    T.zw_hi = zw_max + 4.0f * (zw_max - zw_min);
}

// Complete set-up of triangle `id` from the mosaic: HZ_SETUP_OK, or why it produces nothing.
// copy = 0: the triangle as the reference draws it.  copy = 1, 2: only with the opt-in seam wrap (P.seam_period > 0),
// for a triangle that straddles the +-pi seam of the window and is therefore "too wide" as it stands: the same
// triangle with its left-hand vertices moved one period to the right (1), and that moved one period to the left (2)
// -- its two appearances at the right and left edge of a full-circle panorama.
__device__ __forceinline__ int hz_tri_setup(const HzView& P, unsigned int id, int copy, HzTri& T)
{
    int vj[3], vi[3];
    hz_tri_vertices(id, P.N, vj, vi);
    float e[3], n[3];
    HzVtx v[3];
    #pragma unroll
    for(int k = 0; k < 3; k++)
    {
        e[k] = __ldg(P.e_tab + vi[k]);
        n[k] = __ldg(P.n_tab + vj[k]);
        const float z = (float)__ldg(P.mosaic + (size_t)vj[k] * P.pitch + vi[k]);
        hz_project(P, e[k], n[k], z, v[k]);
        if(copy >= 1 && v[k].xn < 0.0f) v[k].xn += P.seam_period;
        if(copy == 2) v[k].xn -= P.seam_period;
    }
    const int st = hz_tri_bounds(P, v[0], v[1], v[2], T);
    if(st != HZ_SETUP_OK) return st;
    T.id = id;
    hz_tri_planes(P, T, e[0], n[0], v[0].z, e[1], n[1], v[1].z, e[2], n[2], v[2].z);
    // every fragment's depth lies in [zw_lo, zw_hi] (F6): entirely in front of the near plane or behind the far
    // plane means every fragment is clipped (F5).  This removes the giants right under the eye.
    if(T.zw_hi < 0.0f || T.zw_lo > 1.0f) return HZ_SETUP_NOTHING;
    return HZ_SETUP_OK;
}

// The copies of a triangle to draw: 0 always; 1 and 2 if 0 came out too wide and the seam wrap is on.  Usage:
//   for(int copy = 0; copy >= 0; copy = hz_next_copy(P, copy, st)) { st = hz_tri_setup(P, id, copy, T); ... }
__device__ __forceinline__ int hz_next_copy(const HzView& P, int copy, int status_of_copy)
{
    if(copy == 0) return (status_of_copy == HZ_SETUP_TOO_WIDE && P.seam_period > 0.0f) ? 1 : -1;
    return copy == 1 ? 2 : -1;
}

// F7: floor(zw * (2^24-1) + 0.5) for 0 <= zw <= 1, exactly as the double-precision expression of the oracle gives it
// (the product of two 24-bit numbers and the added half are exact in double), in integer arithmetic: B200 has next
// to no FP64 throughput, and this runs once per fragment.
__device__ __forceinline__ unsigned int hz_quantise24(float zw)
{
    const unsigned int bits = __float_as_uint(zw);
    const unsigned int ex = bits >> 23;                      // zw >= 0: no sign bit
    if(ex < 127u - 40u) return 0u;                           // zw < 2^-40: rounds to 0 (also zero and denormals)
    const unsigned long long mant = (unsigned long long)((bits & 0x7FFFFFu) | 0x800000u);
    const unsigned int shift = 150u - ex;                    // zw = mant * 2^-shift, 23 <= shift <= 63
    return (unsigned int)((mant * 16777215ull + (1ull << (shift - 1u))) >> shift);
}

// The depth test: min() into the pixel's key.  P.vis comes out of the shared-memory copy of the parameters, so the
// compiler only knows it as a generic pointer and atomicMin() would become a run-time dispatch on the address space
// with a compare-and-swap loop for the shared-memory case; nothing needs the old value either.  Said explicitly:
// a reduction on a global address (RED.E.MIN.64).
__device__ __forceinline__ void hz_red_min(unsigned long long* p, unsigned long long key)
{
    asm volatile("red.relaxed.gpu.global.min.u64 [%0], %1;" :: "l"(__cvta_generic_to_global(p)), "l"(key) : "memory");
}

// depth test + colour write for one covered pixel centre
__device__ __forceinline__ void hz_fragment(const HzView& P, const HzTri& T, int px, int py)
{
    const float cx = (float)px + 0.5f, cy = (float)py + 0.5f;
    const float ddx = cx - T.xw0, ddy = cy - T.yw0;
    float zw = T.z0w + (T.dzdx * ddx + T.dzdy * ddy);
    zw = fminf(fmaxf(zw, T.zw_lo), T.zw_hi);                                 // F6
    if(!(zw >= 0.0f && zw <= 1.0f)) return;                                  // F5: view-volume clip per fragment
    const unsigned int q = hz_quantise24(zw);                                // F7
    if(q >= HZ_Q_MAX) return;                                                // cannot pass GL_LESS against 1.0
    float r = T.r0 + (T.drdx * ddx + T.drdy * ddy);
    r = fmaxf(fminf(r, 1.0f), 0.0f);
    const unsigned int r8 = (unsigned int)(r * 255.0f + 0.5f);              // F8
    const unsigned long long key = ((unsigned long long)((P.epoch << 24) | q) << HZ_KEY_Q_SHIFT) |
                                   ((unsigned long long)(T.id & HZ_ID_CELL_MASK) << 8) | r8;
    hz_red_min(&P.vis[(size_t)py * (size_t)(P.x1 - P.x0) + (size_t)(px - P.x0)], key);
}

// Edge functions E_k(P) = dx_k*(Py - Y_k) - dy_k*(Px - X_k) on the snapped positions (F3); an edge owns its
// boundary iff it runs downwards, or is horizontal running leftwards (F4).  I = int when every term fits in
// 32 bits (triangle smaller than 64 pixels), long long otherwise.
template <typename I>
struct HzEdges
{
    I dx0, dy0, dx1, dy1, dx2, dy2;
    I b0, b1, b2;
    __device__ __forceinline__ explicit HzEdges(const HzTri& T)
    {
        dx0 = (I)T.X1 - T.X0; dy0 = (I)T.Y1 - T.Y0;
        dx1 = (I)T.X2 - T.X1; dy1 = (I)T.Y2 - T.Y1;
        dx2 = (I)T.X0 - T.X2; dy2 = (I)T.Y0 - T.Y2;
        b0 = (dy0 < 0 || (dy0 == 0 && dx0 < 0)) ? 0 : 1;
        b1 = (dy1 < 0 || (dy1 == 0 && dx1 < 0)) ? 0 : 1;
        b2 = (dy2 < 0 || (dy2 == 0 && dx2 < 0)) ? 0 : 1;
    }
    __device__ __forceinline__ bool inside(const HzTri& T, int px, int py) const
    {
        const I Px = (I)px * 256 + 128, Py = (I)py * 256 + 128;
        const I E0 = dx0 * (Py - T.Y0) - dy0 * (Px - T.X0);
        const I E1 = dx1 * (Py - T.Y1) - dy1 * (Px - T.X1);
        const I E2 = dx2 * (Py - T.Y2) - dy2 * (Px - T.X2);
        return E0 >= b0 && E1 >= b1 && E2 >= b2;
    }
    // true if no pixel centre of the box [px0,px1] x [py0,py1] can be inside: some edge function is below its
    // threshold even at the corner of the box where it is largest
    __device__ __forceinline__ bool box_outside(const HzTri& T, int px0, int px1, int py0, int py1) const
    {
        const I Xa = (I)px0 * 256 + 128, Xb = (I)px1 * 256 + 128;
        const I Ya = (I)py0 * 256 + 128, Yb = (I)py1 * 256 + 128;
        const I M0 = dx0 * ((dx0 > 0 ? Yb : Ya) - T.Y0) - dy0 * ((dy0 > 0 ? Xa : Xb) - T.X0);
        const I M1 = dx1 * ((dx1 > 0 ? Yb : Ya) - T.Y1) - dy1 * ((dy1 > 0 ? Xa : Xb) - T.X1);
        const I M2 = dx2 * ((dx2 > 0 ? Yb : Ya) - T.Y2) - dy2 * ((dy2 > 0 ? Xa : Xb) - T.X2);
        return M0 < b0 || M1 < b1 || M2 < b2;
    }
};

__device__ __forceinline__ bool hz_tri_is_small(const HzTri& T)
{
    const int bx0 = min(min(T.X0, T.X1), T.X2), bx1 = max(max(T.X0, T.X1), T.X2);
    const int by0 = min(min(T.Y0, T.Y1), T.Y2), by1 = max(max(T.Y0, T.Y1), T.Y2);
    return (bx1 - bx0) < 16384 && (by1 - by0) < 16384;      // every difference < 2^14 => products < 2^28, sums and steps far from 2^31
}

// ================================================================================================
// culling pyramid (init)
// ================================================================================================

__global__ void __launch_bounds__(256)
k_minmax_blocks(const int16_t* __restrict__ mosaic, int N, int pitch, short2* __restrict__ mm, int nb)
{
    const int bi = blockIdx.x * blockDim.x + threadIdx.x, bj = blockIdx.y;
    if(bi >= nb) return;
    const int c0 = bi * HZ_BLOCK_CELLS, r0 = bj * HZ_BLOCK_CELLS;
    int lo = 32767, hi = -32768;
    for(int r = r0; r <= min(r0 + HZ_BLOCK_CELLS, N - 1); r++)
        for(int c = c0; c <= min(c0 + HZ_BLOCK_CELLS, N - 1); c++)
        {
            const int z = mosaic[(size_t)r * pitch + c];
            lo = min(lo, z); hi = max(hi, z);
        }
    mm[(size_t)bj * nb + bi] = make_short2((short)lo, (short)hi);
}

__global__ void __launch_bounds__(256)
k_minmax_tiles(const short2* __restrict__ mm, int nb, short2* __restrict__ mt, int nt)
{
    const int ti = blockIdx.x * blockDim.x + threadIdx.x, tj = blockIdx.y;
    if(ti >= nt) return;
    int lo = 32767, hi = -32768;
    for(int r = tj * HZ_TILE_BLOCKS; r < min((tj + 1) * HZ_TILE_BLOCKS, nb); r++)
        for(int c = ti * HZ_TILE_BLOCKS; c < min((ti + 1) * HZ_TILE_BLOCKS, nb); c++)
        {
            const short2 v = mm[(size_t)r * nb + c];
            lo = min(lo, (int)v.x); hi = max(hi, (int)v.y);
        }
    mt[(size_t)tj * nt + ti] = make_short2((short)lo, (short)hi);
}

cudaError_t hz_launch_pyramid(const int16_t* mosaic, int N, int pitch, short2* mm_block, int nb,
                              short2* mm_tile, int nt, cudaStream_t stream)
{
    k_minmax_blocks<<<dim3((nb + 255) / 256, nb), 256, 0, stream>>>(mosaic, N, pitch, mm_block, nb);
    k_minmax_tiles<<<dim3((nt + 255) / 256, nt), 256, 0, stream>>>(mm_block, nb, mm_tile, nt);
    return cudaGetLastError();
}

// ================================================================================================
// conservative tests on rectangles of the mesh
// ================================================================================================
//
// A rectangle of vertices (columns c_lo..c_hi, rows r_lo..r_hi, heights within [zmin,zmax]) is dropped when no
// triangle inside it can produce a fragment that survives:
//   * every vertex is horizontally farther than zfar   -> every fragment fails the far clip
//   * the screen-space box of its vertices holds no pixel centre of the target
//   * every pixel of that box already holds a key with a smaller depth than anything inside can produce
// All three only ever remove work, never a winning fragment, so the image does not depend on them (nor on the
// order in which the visibility buffer fills up).
//
// Screen box.  Inside one quadrant around the eye the azimuth atan2(e,n) is monotonic in e and in n, so its
// extremes over the rectangle sit on two known corners; the elevation atan(h/d) is bounded by the extreme heights
// over the nearest/farthest horizontal distance.  The same device functions as for real vertices are used and
// P.box_margin (1/64 pixel, plus a few float ulps of the largest window coordinate) is added all around, which
// covers their few-ulp non-monotonicity and the 1/512 pixel of snapping.
// Depth.  A vertex depth is a monotonic float function of its slant range >= its horizontal distance >= the
// rectangle's nearest horizontal distance.  A fragment's depth stays within its triangle's vertex depths widened
// by 4x their extent (F6), and the slant ranges of one triangle's vertices differ by at most their 3-D distance
// <= sqrt(cell diagonal^2 + (zmax-zmin)^2).  That gives a lower bound for the depth of every fragment.


struct HzBox { int px0, px1, py0, py1; unsigned int qmin; };
enum { HZ_RECT_DEAD_FAR = 0, HZ_RECT_DEAD_WINDOW = 1, HZ_RECT_ALIVE = 2, HZ_RECT_BOXED = 3 };

__device__ __forceinline__ float hz_window_x(const HzView& P, float e, float n, float halfW)
{
    float az = hz_atan2_az(e, n);
    const float t = (az - P.az_center) * 0.15915494309189535f;
    az = (t - rintf(t)) * 2.f * HZ_PI_F + P.az_center;
    return (az - P.az_center) * P.az_ndc_per_rad * halfW + halfW;
}

__device__ __forceinline__ int
hz_rect_test(const HzView& P, int c_lo, int c_hi, int r_lo, int r_hi, float zmin, float zmax, HzBox& B)
{
    const float e_lo = __ldg(P.e_tab + c_lo), e_hi = __ldg(P.e_tab + c_hi);
    const float n_lo = __ldg(P.n_tab + r_lo), n_hi = __ldg(P.n_tab + r_hi);
    const bool  e_in = (e_lo <= 0.f && e_hi >= 0.f), n_in = (n_lo <= 0.f && n_hi >= 0.f);
    const float e_near = e_in ? 0.f : fminf(fabsf(e_lo), fabsf(e_hi));
    const float n_near = n_in ? 0.f : fminf(fabsf(n_lo), fabsf(n_hi));
    const float d2min = e_near * e_near + n_near * n_near;

    // lower bound of the window depth of any fragment: the nearest corner evaluated like a vertex on the eye's
    // ground plane (hz_depth_shade), minus the extrapolation allowance.  Approximate square roots and a reciprocal
    // instead of the exact operations of a real vertex: each is within 2 ulp, the 2e-5 below (3 m at 150 km) is
    // two orders of magnitude more than they and the later float->integer truncation can add up to.
    {
        const float len = d2min * rsqrtf(fmaxf(d2min, 1e-30f));
        const float dz  = zmax - zmin;
        const float s2  = P.cell_diag2 + dz * dz;
        const float sep = s2 * rsqrtf(s2);
        const float lo  = (len - P.znear - 4.004f * sep) * P.inv_zrange - 2e-5f;
        if(lo > 1.0f) return HZ_RECT_DEAD_FAR;             // every fragment fails the far clip
        B.qmin = (P.epoch << 24) | ((lo <= 0.0f) ? 0u : (unsigned int)(lo * 16777215.0f));    // as hz_key_top() gives it
    }
    if(e_in || n_in) return HZ_RECT_ALIVE;                 // touches an axis through the eye: not worth a box

    const float halfW = 0.5f * (float)P.W, halfH = 0.5f * (float)P.H;
    const bool east = e_lo > 0.f, north = n_lo > 0.f;
    // d(az)/de = n/d^2, d(az)/dn = -e/d^2
    const float x_hi = hz_window_x(P, north ? e_hi : e_lo, east ? n_lo : n_hi, halfW);
    const float x_lo = hz_window_x(P, north ? e_lo : e_hi, east ? n_hi : n_lo, halfW);
    if(!(x_lo <= x_hi)) return HZ_RECT_ALIVE;              // the +-pi seam of the window runs through it

    const float e_far = fmaxf(fabsf(e_lo), fabsf(e_hi)), n_far = fmaxf(fabsf(n_lo), fabsf(n_hi));
    const float d2max = e_far * e_far + n_far * n_far;
    // (with the opt-in earth curvature every height drops by curvature*d^2: by at least that of the nearest and at
    // most that of the farthest point)
    const float hmax = zmax - P.viewer_z - P.curvature * d2min, hmin = zmin - P.viewer_z - P.curvature * d2max;
    const float el_hi = hz_atan_el(hmax, hmax > 0.f ? d2min : d2max);
    const float el_lo = hz_atan_el(hmin, hmin > 0.f ? d2max : d2min);
    const float y_hi = el_hi * P.aspect * P.az_ndc_per_rad * halfH + halfH;
    const float y_lo = el_lo * P.aspect * P.az_ndc_per_rad * halfH + halfH;

    // pixel centres p + 0.5 inside [lo - margin, hi + margin]; the float->int conversions saturate
    const float fx0 = ceilf(x_lo - 0.5f - P.box_margin), fx1 = floorf(x_hi - 0.5f + P.box_margin);
    const float fy0 = ceilf(y_lo - 0.5f - P.box_margin), fy1 = floorf(y_hi - 0.5f + P.box_margin);
    if(!(fx0 <= fx1 && fy0 <= fy1)) return HZ_RECT_DEAD_WINDOW;
    if(fx1 < (float)P.x0 || fx0 > (float)(P.x1 - 1) || fy1 < 0.f || fy0 > (float)(P.H - 1)) return HZ_RECT_DEAD_WINDOW;
    B.px0 = max((int)fx0, P.x0); B.px1 = min((int)fx1, P.x1 - 1);
    B.py0 = max((int)fy0, 0);    B.py1 = min((int)fy1, P.H - 1);
    return HZ_RECT_BOXED;
}

// ================================================================================================
// exact stages for one block of 4x4 cells: projection, integer cull, set-up, rasterisation
// ================================================================================================

#define HZ_WARPS_PER_CTA 8
#ifndef HZ_MESH_CTAS
#define HZ_MESH_CTAS 4             /* resident CTAs per SM the meshing kernels are compiled for (register budget) */
#endif
#ifndef HZ_BIG_ROWS
#define HZ_BIG_ROWS      16        /* large bounding boxes are cut into sub-boxes of this size for k_big (4 and 8 rows: */
#endif                             /* the per-sub-box set-up weighs more, measured slower in zoomed-in views and batches): */
#define HZ_BIG_COLS      32        /* lane = column, a few rows each (more for very large triangles) */
#define HZ_BIG_MAX_ENTRIES 64u
#define HZ_MID_LANES     16        /* lanes of a warp with a middle-sized triangle from which on they draw them themselves */
#define HZ_BIG_RECOMPUTE   0x80000000u   /* queue entry: .x is a triangle number (set up again), not a record */

struct HzLaneVtx { int X, Y; };

__device__ __forceinline__ HzLaneVtx hz_lane_vertex(const HzView& P, float e, float n, float z, float halfW, float halfH)
{
    HzVtx v;
    hz_project(P, e, n, z, v);
    HzLaneVtx o;
    o.X = hz_snap(v.xn * halfW + halfW);
    o.Y = hz_snap(v.yn * halfH + halfH);
    return o;
}

// the rasteriser's integer tests for one triangle (hz_tri_bounds without the float-only seam/guard tests,
// which set-up applies; a triangle that fails here cannot produce a fragment there).  [x0, x1) x [0, H) = the target;
// wide: see below.
__device__ __forceinline__ bool
hz_tri_alive(int x0, int x1, int H, int wide, const HzLaneVtx& a, const HzLaneVtx& b, const HzLaneVtx& c)
{
    const int bx0 = min(min(a.X, b.X), c.X), bx1 = max(max(a.X, b.X), c.X);
    const int by0 = min(min(a.Y, b.Y), c.Y), by1 = max(max(a.Y, b.Y), c.Y);
    const int px0 = max((bx0 + 127) >> 8, x0), px1 = min((bx1 - 128) >> 8, x1 - 1);
    const int py0 = max((by0 + 127) >> 8, 0),  py1 = min((by1 - 128) >> 8, H - 1);
    if(px0 > px1 || py0 > py1) return false;            // no pixel centre of the target inside the bounding box
    // opt-in seam wrap (wide = W * 64 - 1024 in 1/256 pixel, else never): a triangle about a quarter of the window
    // wide or more may be a seam straddler whose two copies show at the edges; its facing as it stands says nothing,
    // set-up decides
    if(bx1 - bx0 >= wide) return true;
    const long long area = (long long)(b.X - a.X) * (c.Y - a.Y) - (long long)(c.X - a.X) * (b.Y - a.Y);
    return area > 0;
}

// one thread walks the whole bounding box; the edge functions are stepped (E(x+1) = E(x) - 256*dy, E(y+1) = E(y) + 256*dx)
template <typename I>
__device__ __forceinline__ void hz_draw_box(const HzView& P, const HzTri& T)
{
    const HzEdges<I> E(T);
    const I Px = (I)T.px0 * 256 + 128, Py = (I)T.py0 * 256 + 128;
    I r0 = E.dx0 * (Py - T.Y0) - E.dy0 * (Px - T.X0) - E.b0;      // >= 0 <=> inside, per edge
    I r1 = E.dx1 * (Py - T.Y1) - E.dy1 * (Px - T.X1) - E.b1;
    I r2 = E.dx2 * (Py - T.Y2) - E.dy2 * (Px - T.X2) - E.b2;
    const I sx0 = E.dy0 * 256, sx1 = E.dy1 * 256, sx2 = E.dy2 * 256;
    const I sy0 = E.dx0 * 256, sy1 = E.dx1 * 256, sy2 = E.dx2 * 256;
    for(int py = T.py0; py <= T.py1; py++)
    {
        I e0 = r0, e1 = r1, e2 = r2;
        for(int px = T.px0; px <= T.px1; px++)
        {
            if((e0 | e1 | e2) >= 0) hz_fragment(P, T, px, py);
            e0 -= sx0; e1 -= sx1; e2 -= sx2;
        }
        r0 += sy0; r1 += sy1; r2 += sy2;
    }
}

// Never on the normal path: draws one triangle completely, whatever its size, in the calling thread.  Used when a
// queue is full.  Kept out of line so that its registers (64-bit edge functions) spill here instead of inflating
// the kernels that merely might call it.
// only_copy < 0: every copy that applies (see hz_tri_setup); else just that one.
__device__ __noinline__ void hz_draw_slow(const HzView& P, unsigned int id, int only_copy)
{
    int st = HZ_SETUP_NOTHING;
    for(int copy = max(only_copy, 0); copy >= 0; copy = (only_copy < 0) ? hz_next_copy(P, copy, st) : -1)
    {
        HzTri T;
        st = hz_tri_setup(P, id, copy, T);
        if(st != HZ_SETUP_OK) continue;
        if(hz_tri_is_small(T)) hz_draw_box<int>(P, T);
        else                   hz_draw_box<long long>(P, T);
    }
}

// What k_big needs of a set-up triangle, as 6 x 16 bytes in the record pool (set-up is ~500 instructions per
// triangle; k_big has one warp per sub-box and would repeat it for each).
#define HZ_TRI_RECORD_VEC 6
__device__ __forceinline__ void hz_tri_store(uint4* rec, const HzTri& T)
{
    rec[0] = make_uint4((unsigned)T.X0, (unsigned)T.Y0, (unsigned)T.X1, (unsigned)T.Y1);
    rec[1] = make_uint4((unsigned)T.X2, (unsigned)T.Y2, (unsigned)T.px0, (unsigned)T.px1);
    rec[2] = make_uint4((unsigned)T.py0, (unsigned)T.py1, __float_as_uint(T.xw0), __float_as_uint(T.yw0));
    rec[3] = make_uint4(__float_as_uint(T.z0w), __float_as_uint(T.r0), __float_as_uint(T.dzdx), __float_as_uint(T.dzdy));
    rec[4] = make_uint4(__float_as_uint(T.drdx), __float_as_uint(T.drdy), __float_as_uint(T.zw_lo), __float_as_uint(T.zw_hi));
    rec[5] = make_uint4(T.id, 0u, 0u, 0u);
}
__device__ __forceinline__ void hz_tri_load(const uint4* rec, HzTri& T)
{
    const uint4 a = __ldcg(rec + 0), b = __ldcg(rec + 1), c = __ldcg(rec + 2), d = __ldcg(rec + 3), e = __ldcg(rec + 4),
                f = __ldcg(rec + 5);
    T.X0 = (int)a.x; T.Y0 = (int)a.y; T.X1 = (int)a.z; T.Y1 = (int)a.w;
    T.X2 = (int)b.x; T.Y2 = (int)b.y; T.px0 = (int)b.z; T.px1 = (int)b.w;
    T.py0 = (int)c.x; T.py1 = (int)c.y; T.xw0 = __uint_as_float(c.z); T.yw0 = __uint_as_float(c.w);
    T.z0w = __uint_as_float(d.x); T.r0 = __uint_as_float(d.y); T.dzdx = __uint_as_float(d.z); T.dzdy = __uint_as_float(d.w);
    T.drdx = __uint_as_float(e.x); T.drdy = __uint_as_float(e.y); T.zw_lo = __uint_as_float(e.z); T.zw_hi = __uint_as_float(e.w);
    T.id = f.x;
}

// How a set-up triangle is drawn: by the thread that set it up if its bounding box has at most P.small_max_pix pixels
// and 32-bit edge functions do, otherwise by k_big, one warp per sub-box of HZ_BIG_COLS columns x (HZ_BIG_ROWS << k)
// rows -- k the smallest that keeps the number of queue entries of the triangle (written by one thread) at or below
// HZ_BIG_MAX_ENTRIES where possible.  Returns the number of sub-boxes, 0 = draw it yourself.
__device__ __forceinline__ unsigned int hz_big_layout(const HzView& P, const HzTri& T, unsigned int& nx, unsigned int& k)
{
    const int bw = T.px1 - T.px0 + 1, bh = T.py1 - T.py0 + 1;
    if(bw * bh <= P.small_max_pix && hz_tri_is_small(T)) return 0;
    nx = (unsigned int)((bw + HZ_BIG_COLS - 1) / HZ_BIG_COLS);
    k = 0;
    unsigned int ny = (unsigned int)((bh + HZ_BIG_ROWS - 1) / HZ_BIG_ROWS);
    while(nx * ny > HZ_BIG_MAX_ENTRIES && ny > 1) { k++; ny = (unsigned int)((bh + (HZ_BIG_ROWS << k) - 1) / (HZ_BIG_ROWS << k)); }
    return nx * ny;
}

// Queues a large triangle: `slot` = first of its n = nx*ny reserved queue slots, `rec` = its reserved record.  False if
// the queue is full: the reserved slots are poisoned (k_big skips those) and the caller has to draw the triangle itself
// (hz_draw_slow; not from here: that call in the middle of k_raster's loop cost it 16 registers and spills).
__device__ __forceinline__ bool
hz_big_enqueue(const HzView& P, const HzTri& T, unsigned int id, int copy, unsigned int nx, unsigned int k, unsigned int n,
               unsigned int slot, unsigned int rec)
{
    if(slot + n > P.big_capacity)
    {
        for(unsigned int q = slot; q < min(slot + n, P.big_capacity); q++) P.big_queue[q] = make_uint2(0xFFFFFFFFu, 0u);
        return false;
    }
    // the set-up triangle goes to the record pool; if that is full the entries carry the triangle's number instead and
    // k_big repeats the set-up (slower, still one warp per sub-box)
    unsigned int first = rec, tag = k << 24;
    if(rec < P.bigtri_capacity) hz_tri_store(P.bigtri + (size_t)rec * HZ_TRI_RECORD_VEC, T);
    else { first = id; tag |= HZ_BIG_RECOMPUTE | ((unsigned int)copy << 28); }
    const unsigned int ny = n / nx;
    for(unsigned int by = 0; by < ny; by++)
        for(unsigned int bx = 0; bx < nx; bx++)
            P.big_queue[slot + by * nx + bx] = make_uint2(first, by | (bx << 12) | tag);
    return true;
}

// The two seam copies of a triangle that came out too wide (opt-in seam wrap; rare): one thread does it all, with
// its own reservations.  Returns the number of queue entries made.
__device__ __noinline__ unsigned int hz_raster_seam_copies(const HzView& P, unsigned int id)
{
    unsigned int queued = 0;
    for(int copy = 1; copy <= 2; copy++)
    {
        HzTri T;
        if(hz_tri_setup(P, id, copy, T) != HZ_SETUP_OK) continue;
        unsigned int nx = 0, k = 0;
        const unsigned int n = hz_big_layout(P, T, nx, k);
        if(n == 0) { hz_draw_box<int>(P, T); continue; }
        const unsigned int slot = atomicAdd(P.big_count, n), rec = atomicAdd(P.bigtri_count, 1u);
        if(hz_big_enqueue(P, T, id, copy, nx, k, n, slot, rec)) queued += n;
        else hz_draw_slow(P, id, copy);
    }
    return queued;
}

// k_raster's rare cases for one triangle: the large-triangle queue was full -> drawn by this thread, whatever its size;
// too wide as it stands and the opt-in seam wrap is on -> its two seam copies.  Returns the queue entries made.
__device__ __noinline__ unsigned int hz_raster_rare(const HzView& P, unsigned int id, int status)
{
    if(status == HZ_SETUP_QUEUE_FULL) { hz_draw_slow(P, id, 0); return 0; }
    if(status == HZ_SETUP_TOO_WIDE && P.seam_period > 0.0f) return hz_raster_seam_copies(P, id);
    return 0;
}

__device__ __forceinline__ unsigned int hz_warp_sum(unsigned int v)
{
    #pragma unroll
    for(int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// A warp meshes HZ_MESH_GROUP blocks per trip: their 5x5 vertices are projected as ONE list of up to 125, in 4 rounds
// of 32 lanes (a block at a time would leave 7 of 32 lanes idle while its 25 vertices are projected, and pay the
// loop's fixed cost five times), then each block's 32 triangles are tested with lane = triangle.
#define HZ_MESH_GROUP  5
#define HZ_MESH_ROUNDS 4           /* ceil(5 * 25 / 32) */
#define HZ_STAGE_SLOTS 64          /* < 32 pending + at most 32 new per block */
struct HzMeshWarp
{
    HzLaneVtx    verts[HZ_MESH_GROUP * 25];
    unsigned int stage[HZ_STAGE_SLOTS];       // triangles that passed the exact tests, not yet in the stage's list
};

// Which vertex a lane handles in each round of a group, worked out once per kernel: vertex v = 32 * round + lane is
// vertex (r, c) of the 5x5 of block k = v / 25 of the group, packed as k | r << 8 | c << 16 (k = 7: none).
struct HzLaneMap { unsigned int code[HZ_MESH_ROUNDS]; };

__device__ __forceinline__ HzLaneMap hz_lane_map(int lane)
{
    HzLaneMap m;
    #pragma unroll
    for(int round = 0; round < HZ_MESH_ROUNDS; round++)
    {
        const int v = round * 32 + lane, k = v / 25, idx = v - 25 * k, r = idx / 5, c = idx - 5 * r;
        m.code[round] = k < HZ_MESH_GROUP ? (unsigned int)(k | (r << 8) | (c << 16)) : 7u;
    }
    return m;
}

// Mesh row vj and column vi of the vertex `code` stands for (blocks are bj << 16 | bi; lane k of `ids` holds block k
// of the group); false beyond the group's last vertex.  All lanes call.  The mosaic and the axis tables are padded
// (HZ_MESH_PAD), so the vertices of blocks that hang over the mesh's last row/column need no clamping: their triangles
// are left out later.
__device__ __forceinline__ bool hz_group_vertex(unsigned int ids, int nblk, unsigned int code, int lod, int& vj, int& vi)
{
    const int k = (int)(code & 7u);
    const unsigned int id = __shfl_sync(0xffffffffu, ids, k);
    vj = ((int)(id >> 16) * HZ_BLOCK_CELLS + (int)((code >> 8) & 7u)) << lod;
    vi = ((int)(id & 0xFFFFu) * HZ_BLOCK_CELLS + (int)(code >> 16)) << lod;
    return k < nblk;
}

// heights of the vertices this lane projects for a group: fetched apart from the meshing so that the caller can have
// the next group's DRAM reads in flight while it works on the current one
struct HzGroupZ { float z[HZ_MESH_ROUNDS]; };

__device__ __forceinline__ HzGroupZ hz_group_heights(const HzView& P, unsigned int ids, int nblk, const HzLaneMap& map)
{
    HzGroupZ g;
    const int16_t* mosaic = P.mosaic;
    const unsigned int pitch = (unsigned int)P.pitch;
    const int lod = P.lod;
    #pragma unroll
    for(int round = 0; round < HZ_MESH_ROUNDS; round++)
    {
        int vj, vi;
        g.z[round] = hz_group_vertex(ids, nblk, map.code[round], lod, vj, vi)
                         ? (float)__ldg(mosaic + (unsigned int)vj * pitch + (unsigned int)vi) : 0.f;
    }
    return g;
}

// Writes stage[0..count) to the triangle list with one atomic; all lanes call.  Returns how many did NOT fit (list
// full): those are moved to the front of the stage, and the caller stops staging and draws them itself (hz_mesh_slow).
// No call to the slow path from here: a call inside the meshing loop makes ptxas keep that loop's registers in local
// memory around it.
__device__ __forceinline__ int hz_stage_flush(const HzView& P, unsigned int* stage, int count, int lane)
{
    if(count == 0) return 0;
    unsigned int base = 0;
    if(lane == 0) base = atomicAdd(P.tri_count, (unsigned int)count);
    base = __shfl_sync(0xffffffffu, base, 0);
    const int fits = (int)min((unsigned int)count, P.tri_capacity - min(base, P.tri_capacity));
    for(int k = lane; k < fits; k += 32) P.tri_queue[base + k] = stage[k];
    if(fits == count) return 0;
    __syncwarp();
    // (count <= 64: two strided passes move the rest down without overlap problems, reads before writes)
    const unsigned int m0 = (fits + lane < count) ? stage[fits + lane] : 0u, m1 = (fits + 32 + lane < count) ? stage[fits + 32 + lane] : 0u;
    __syncwarp();
    if(fits + lane < count) stage[lane] = m0;
    if(fits + 32 + lane < count) stage[32 + lane] = m1;
    __syncwarp();
    return count - fits;
}

// Projects the vertices of the group's nblk blocks (ids / Z as above) into M.verts.  All lanes call.
__device__ __forceinline__ void
hz_group_project(const HzView& P, unsigned int ids, int nblk, int lane, const HzLaneMap& map, const HzGroupZ& Z, HzMeshWarp& M)
{
    const float halfW = 0.5f * (float)P.W, halfH = 0.5f * (float)P.H;
    const float* e_tab = P.e_tab;
    const float* n_tab = P.n_tab;
    const int lod = P.lod;
    #pragma unroll 1            // one projection's registers at a time (unrolled, ptxas interleaves the four and spills)
    for(int round = 0; round < HZ_MESH_ROUNDS; round++)
    {
        int vj, vi;
        const float z = round == 0 ? Z.z[0] : round == 1 ? Z.z[1] : round == 2 ? Z.z[2] : Z.z[3];
        const unsigned int code = round == 0 ? map.code[0] : round == 1 ? map.code[1] : round == 2 ? map.code[2] : map.code[3];
        if(hz_group_vertex(ids, nblk, code, lod, vj, vi))
            M.verts[round * 32 + lane] = hz_lane_vertex(P, __ldg(e_tab + vi), __ldg(n_tab + vj), z, halfW, halfH);
    }
    __syncwarp();
}

// The triangles of blocks k0 .. nblk-1 of a projected group, lane = triangle: the numbers of those that pass the exact
// integer tests go to the warp's stage, which is written to the stage's triangle list whenever it holds 32 or more
// (`count` = the stage's fill, the same in all lanes; `passed` counts them).  Returns -1 -- or, if the list turned
// out to be full, the block to resume at (<= nblk): the stage then holds `count` (< 64) triangles that the caller must
// draw itself, and it goes on with SLOW = true, where every triangle that passes is drawn on the spot (hz_draw_slow).  That
// call is kept out of the fast variant: a call inside the meshing loop makes ptxas keep the loop's registers in local
// memory around it.
template <bool SLOW>
__device__ __forceinline__ int
hz_group_triangles(const HzView& P, unsigned int ids, int k0, int nblk, int lane, HzMeshWarp& M, int& count, unsigned int& passed)
{
    // (copies: P lives in shared memory like M, and every store to M would make the compiler read these again)
    const int N1 = P.N - 1, x0 = P.x0, x1 = P.x1, H = P.H, lod = P.lod;
    const int wide = P.seam_period > 0.0f ? P.W * 64 - 1024 : 0x7FFFFFFF;      // see hz_tri_alive
    const int jmax = N1 - (1 << lod);                                           // last row/column a triangle may start at
    // cell (cr, cc) of the block, its lower-left vertex a, upper-right vertex d, and the third one
    // lib:496-508: even triangle (j,i),(j+1,i+1),(j+1,i) ; odd triangle (j,i),(j,i+1),(j+1,i+1)
    const int cell = lane >> 1, cr = cell >> 2, cc = cell & 3;
    const bool odd = (lane & 1) != 0;
    const int ia = cr * 5 + cc, id_ = ia + 6, io = odd ? ia + 1 : ia + 5;
    for(int k = k0; k < nblk; k++)
    {
        const unsigned int id = __shfl_sync(0xffffffffu, ids, k);
        const int j = ((int)(id >> 16) * HZ_BLOCK_CELLS + cr) << lod, i = ((int)(id & 0xFFFFu) * HZ_BLOCK_CELLS + cc) << lod;
        // (one evaluation with selected operands: under an odd/even branch each half would run with half the lanes)
        const HzLaneVtx* vb = M.verts + 25 * k;
        const HzLaneVtx a = vb[ia], d = vb[id_], o = vb[io];
        const bool on = j <= jmax && i <= jmax && hz_tri_alive(x0, x1, H, wide, a, odd ? o : d, odd ? d : o);
        const unsigned int ballot = __ballot_sync(0xffffffffu, on);
        if(ballot == 0) continue;
        const unsigned int tri = (2u * ((unsigned int)j * (unsigned int)N1 + (unsigned int)i) + (unsigned int)(lane & 1)) |
                                 ((unsigned int)lod << HZ_ID_LOD_SHIFT);
        passed += (unsigned int)__popc(ballot);
        if(SLOW)
        {
            if(on) hz_draw_slow(P, tri, -1);
            continue;
        }
        if(on) M.stage[count + __popc(ballot & ((1u << lane) - 1u))] = tri;
        count += __popc(ballot);
        __syncwarp();
        if(count >= 32)
        {
            count = hz_stage_flush(P, M.stage, count, lane);
            __syncwarp();
            if(count > 0) return k + 1;         // list full
        }
    }
    return -1;
}

// What a meshing warp does once the stage's list is full (never on the normal path): draws what is staged.
__device__ __noinline__ void hz_stage_draw_slow(const HzView& P, const unsigned int* stage, int count)
{
    for(int q = (int)(threadIdx.x & 31u); q < count; q += 32) hz_draw_slow(P, stage[q], -1);
}

// end of a meshing kernel: the leftovers of all warps of the CTA go out with one atomic.  Every thread calls.
__device__ __forceinline__ void
hz_stage_flush_cta(const HzView& P, const HzMeshWarp& M, int count, unsigned int* s_total, unsigned int* s_base)
{
    const int lane = threadIdx.x & 31;
    if(threadIdx.x == 0) *s_total = 0;
    __syncthreads();
    unsigned int off = 0;
    if(lane == 0 && count) off = atomicAdd(s_total, (unsigned int)count);
    off = __shfl_sync(0xffffffffu, off, 0);
    __syncthreads();
    const unsigned int total = *s_total;
    if(total == 0) return;
    if(threadIdx.x == 0) *s_base = atomicAdd(P.tri_count, total);
    __syncthreads();
    const unsigned int base = *s_base + off;
    for(int k = lane; k < count; k += 32)
    {
        if(base + k < P.tri_capacity) P.tri_queue[base + k] = M.stage[k];
        else                          hz_draw_slow(P, M.stage[k], -1);     // list full; after the meshing loop, so harmless
    }
}

// What a meshing warp does from the moment the stage's triangle list is full (never on the normal path; tests shrink
// the list to get here): it draws what it has staged, then meshes the rest of its blocks with every passing triangle
// drawn on the spot.  One out-of-line function with its own register allocation, called once at the end of the kernel:
// inlined, its calls to hz_draw_slow() made ptxas keep the hot meshing loop's registers in local memory.
// b: first block of the group the warp stopped in (already projected, to be resumed at block k_resume), ids: that
// group's blocks; the warp's later groups start `stride` blocks on.  near: k_near's blocks are not queued but counted
// off a rectangle of the block grid (G), k_mesh's come from P.block_queue (G = null).
struct HzNearGrid { int bj0, bi0, nbi; };

__device__ __noinline__ void
hz_mesh_slow_tail(const HzView& P, HzMeshWarp& M, int staged, unsigned int b, unsigned int n, unsigned int stride, int per,
                  unsigned int ids, int k_resume, const HzNearGrid* G, unsigned int& n_meshed, unsigned int& n_tris)
{
    const int lane = (int)(threadIdx.x & 31u);
    const HzLaneMap map = hz_lane_map(lane);
    hz_stage_draw_slow(P, M.stage, staged);
    int count = 0;
    for(bool first = true; b < n; b += stride, first = false)
    {
        const int nblk = (int)min((unsigned int)per, n - b);
        if(!first)
        {
            if(G != nullptr)
            {
                const int bk = (int)min(b + (unsigned int)lane, n - 1u);
                ids = ((unsigned int)(G->bj0 + bk / G->nbi) << 16) | (unsigned int)(G->bi0 + bk % G->nbi);
            }
            else ids = (b + lane < n && lane < per) ? P.block_queue[b + lane] : 0u;
            hz_group_project(P, ids, nblk, lane, map, hz_group_heights(P, ids, nblk, map), M);
            n_meshed += (unsigned int)nblk;
        }
        hz_group_triangles<true>(P, ids, first ? k_resume : 0, nblk, lane, M, count, n_tris);
        __syncwarp();
    }
}

// ================================================================================================
// k_near: the tiles around the eye, one warp per block, no pyramid and no occlusion tests
// ================================================================================================

__device__ __forceinline__ void hz_near_tiles(const HzView& P, int& ti0, int& ti1, int& tj0, int& tj1)
{
    ti0 = max(P.eye_ti - P.near_rings, 0); ti1 = min(P.eye_ti + P.near_rings, P.nt - 1);
    tj0 = max(P.eye_tj - P.near_rings, 0); tj1 = min(P.eye_tj + P.near_rings, P.nt - 1);
}

__global__ void __launch_bounds__(HZ_WARPS_PER_CTA * 32, HZ_MESH_CTAS)
k_near(const HzView* __restrict__ V)
{
    HZ_KERNEL_PROLOGUE(V, P);
    __shared__ HzMeshWarp s_warp[HZ_WARPS_PER_CTA];
    __shared__ unsigned int s_total, s_base;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const HzLaneMap map = hz_lane_map(lane);

    int ti0, ti1, tj0, tj1;
    hz_near_tiles(P, ti0, ti1, tj0, tj1);
    const int bi0 = ti0 * HZ_TILE_BLOCKS, bi1 = min((ti1 + 1) * HZ_TILE_BLOCKS, P.nb);
    const int bj0 = tj0 * HZ_TILE_BLOCKS, bj1 = min((tj1 + 1) * HZ_TILE_BLOCKS, P.nb);
    const int nbi = bi1 - bi0, nblocks = nbi * (bj1 - bj0);
    const int nwarps = gridDim.x * HZ_WARPS_PER_CTA;
    // no conservative tests here: next to the eye nearly every block shows, and what does not falls to the exact
    // integer tests of hz_mesh_group anyway
    // blocks per warp and trip: as many as a group holds when there is enough work for that, fewer when the warps would
    // otherwise go idle (a lone view: the pass is latency-bound)
    const int per = min(HZ_MESH_GROUP, max(1, (nblocks + nwarps - 1) / nwarps));
    unsigned int n_blocks = 0, n_tris = 0;
    int count = 0, b = (blockIdx.x * HZ_WARPS_PER_CTA + wib) * per, k_resume = -1;
    HzMeshWarp& M = s_warp[wib];
    for(; b < nblocks && k_resume < 0; b += nwarps * per)
    {
        const int nblk = min(per, nblocks - b), bk = min(b + lane, nblocks - 1);
        const unsigned int ids = ((unsigned int)(bj0 + bk / nbi) << 16) | (unsigned int)(bi0 + bk % nbi);
        n_blocks += (unsigned int)nblk;
        hz_group_project(P, ids, nblk, lane, map, hz_group_heights(P, ids, nblk, map), M);
        k_resume = hz_group_triangles<false>(P, ids, 0, nblk, lane, M, count, n_tris);
        __syncwarp();
    }
    if(k_resume >= 0)
    {
        // the triangle list is full: this warp draws everything else it finds itself (b already points at the next
        // group; the one it stopped in is still projected)
        b -= nwarps * per;
        const HzNearGrid G = { bj0, bi0, nbi };
        const int bk = min(b + lane, nblocks - 1);
        const unsigned int ids = ((unsigned int)(bj0 + bk / nbi) << 16) | (unsigned int)(bi0 + bk % nbi);
        hz_mesh_slow_tail(P, M, count, (unsigned int)b, (unsigned int)nblocks, (unsigned int)(nwarps * per), per, ids, k_resume, &G,
                          n_blocks, n_tris);
        count = 0;
    }
    hz_stage_flush_cta(P, s_warp[wib], count, &s_total, &s_base);
    if(P.stats && lane == 0 && n_blocks)
    {
        atomicAdd(P.stats + HZ_STAT_BLOCKS, n_blocks);
        atomicAdd(P.stats + HZ_STAT_BLOCKS_MESHED, n_blocks);
        atomicAdd(P.stats + HZ_STAT_TRIANGLES, n_tris);
    }
}

cudaError_t hz_launch_near(const HzView& v, const HzView* d_v, int nviews, cudaStream_t stream)
{
    const int side = min(2 * v.near_rings + 1, v.nt) * HZ_TILE_BLOCKS;
    const int nblocks = side * side;
    int ctas = (nblocks + HZ_WARPS_PER_CTA - 1) / HZ_WARPS_PER_CTA;      // (k_near fits its group size to the grid)
    const int cap = max(148 * 8 / max(nviews, 1), 37);
    if(ctas > cap) ctas = cap;
    if(ctas < 1) ctas = 1;
    return hz_launch(k_near, dim3(ctas, (unsigned)nviews), dim3(HZ_WARPS_PER_CTA * 32), stream, d_v);
}

// ================================================================================================
// k_tiles / k_blocks / k_mesh: everything beyond the near tiles, hierarchically culled, band by band
// ================================================================================================
//
// The rest of the mesh is walked in a few bands of growing Chebyshev distance (in tiles) around the eye's tile.
// Per band four kernels run back to back, each with one unit of work per thread or warp so that no warp ever
// carries a long serial chain:
//   k_tiles   thread = tile (32x32 cells): conservative test of the whole tile        -> queue of live tiles
//   k_blocks  thread = block (4x4 cells) of a live tile: the same test on the block   -> queue of live blocks
//   k_mesh    warp   = live block: projection, exact integer cull (lane = triangle)   -> list of triangles
//   k_raster  thread = triangle: set-up, rasterisation, depth test
// Everything a band draws is in the visibility buffer before the next band is tested against it, and within a
// band whatever has already been drawn helps too.

// The box is walked along its longer side, HZ_OCCL_FETCH keys per round (so that the L2 round trips overlap: a lone view
// waits for every one of them); only the upper half of a key is fetched -- epoch and depth sit in its top 27 bits --
// and the walk ends at the first round that shows something not nearer.  (The first version walked the box as one run
// of pixels: the wrap to the next row, tested per pixel, cost as much as the fetch and the comparison together.)
#ifndef HZ_OCCL_FETCH
#define HZ_OCCL_FETCH 8            /* (16 and 32 measured no better, lone or batched) */
#endif
__device__ __forceinline__ bool hz_box_occluded_thread(const HzView& P, const HzBox& B, int max_pix)
{
    const int w = B.px1 - B.px0 + 1, h = B.py1 - B.py0 + 1;
    if(w * h > max_pix) return false;
    const unsigned int Wt2 = 2u * (unsigned int)(P.x1 - P.x0);                // 32-bit words per row of keys
    // (upper word of the first key of the box)
    const unsigned int* line = (const unsigned int*)P.vis + ((size_t)B.py0 * Wt2 + 2u * (unsigned int)(B.px0 - P.x0) + 1u);
    const unsigned int qmin_hi = B.qmin << (HZ_KEY_Q_SHIFT - 32);             // the bound, placed like the key's upper word
    const bool rows = w >= h;                                                 // lines = rows of the box, or its columns
    const int n_lines = rows ? h : w, n_along = rows ? w : h;
    const unsigned int step_line = rows ? Wt2 : 2u, step_along = rows ? 2u : Wt2;
    for(int l = 0; l < n_lines; l++, line += step_line)
    {
        const unsigned int* p = line;
        for(int a = 0; a < n_along; a += HZ_OCCL_FETCH, p += HZ_OCCL_FETCH * step_along)
        {
            // all fetches of the round first, none of them conditional (beyond the end of the line the last key is
            // fetched again).  Whether the loads really go out together hangs on ptxas's register heuristics: one
            // build of k_tiles came out with 40 instead of 48 registers, two or three loads in flight instead of
            // eight, and a lone panorama 12 us slower.  The culling kernels therefore say __launch_bounds__(256, 3):
            // with a stated register budget (85) ptxas schedules for the loads, and uses 48 (tools/sass_census.py).
            unsigned int k[HZ_OCCL_FETCH];
            const int last = n_along - 1 - a;
            #pragma unroll
            for(int u = 0; u < HZ_OCCL_FETCH; u++) k[u] = __ldcg(p + (unsigned int)min(u, last) * step_along);
            unsigned int farthest = 0;
            #pragma unroll
            for(int u = 0; u < HZ_OCCL_FETCH; u++) farthest = max(farthest, k[u]);
            // (the upper word holds epoch | depth | the top 5 bits of the triangle number: comparing it whole against
            // the bound with those 5 bits clear is the same test as comparing the top 27 bits)
            if(farthest >= qmin_hi) return false;
        }
    }
    return true;
}

// Appends `value` of every thread with `on` to queue[*count...] with ONE global atomic per CTA: thousands of warps
// bumping the same counter serialise in one L2 slice, which is what these short kernels would otherwise wait on.
// Every thread of the CTA must call it (it synchronises the CTA), with `on` false where there is nothing to add.
struct HzCtaAppend
{
    unsigned int count, base;
    unsigned int buf[256];
};

__device__ __forceinline__ void
hz_cta_append(HzCtaAppend& A, bool on, unsigned int value, unsigned int* queue, unsigned int* count)
{
    const int lane = threadIdx.x & 31;
    if(threadIdx.x == 0) A.count = 0;
    __syncthreads();
    const unsigned int ballot = __ballot_sync(0xffffffffu, on);
    unsigned int wbase = 0;
    if(lane == 0 && ballot) wbase = atomicAdd(&A.count, (unsigned int)__popc(ballot));
    wbase = __shfl_sync(0xffffffffu, wbase, 0);
    if(on) A.buf[wbase + __popc(ballot & ((1u << lane) - 1u))] = value;
    __syncthreads();
    const unsigned int n = A.count;
    if(n == 0) return;                                   // the same for the whole CTA
    if(threadIdx.x == 0) A.base = atomicAdd(count, n);
    __syncthreads();
    if(threadIdx.x < n) queue[A.base + threadIdx.x] = A.buf[threadIdx.x];
}

// diagnostics: per-CTA sums in shared memory, then one global atomic per counter and CTA (only when P.stats is set)
__device__ __forceinline__ void hz_cta_stats4(unsigned int* s4, unsigned int* global4, unsigned int a, unsigned int b,
                                              unsigned int c, unsigned int d)
{
    if(threadIdx.x < 4) s4[threadIdx.x] = 0;
    __syncthreads();
    a = hz_warp_sum(a); b = hz_warp_sum(b); c = hz_warp_sum(c); d = hz_warp_sum(d);
    if((threadIdx.x & 31) == 0) { atomicAdd(s4 + 0, a); atomicAdd(s4 + 1, b); atomicAdd(s4 + 2, c); atomicAdd(s4 + 3, d); }
    __syncthreads();
    if(threadIdx.x < 4 && s4[threadIdx.x]) atomicAdd(global4 + threadIdx.x, s4[threadIdx.x]);
}

__global__ void __launch_bounds__(256, 3)
k_tiles(const HzView* __restrict__ V)
{
    HZ_KERNEL_PROLOGUE(V, P);
    __shared__ HzCtaAppend s_app;
    __shared__ unsigned int s_stats[4];
    const int nt = P.nt, N = P.N;
    const int rmax = max(max(P.eye_ti, nt - 1 - P.eye_ti), max(P.eye_tj, nt - 1 - P.eye_tj));
    const int ring_hi = min(P.ring_hi, rmax + 1), ring_lo = P.ring_lo;
    if(ring_lo >= ring_hi) return;
    // the band = the tiles of Chebyshev distance [ring_lo, ring_hi) from the eye's tile: the threads walk the part of
    // its bounding square that lies inside the mesh, row by row, and skip the hole in the middle
    const int tx0 = max(P.eye_ti - (ring_hi - 1), 0), tx1 = min(P.eye_ti + (ring_hi - 1), nt - 1);
    const int ty0 = max(P.eye_tj - (ring_hi - 1), 0), ty1 = min(P.eye_tj + (ring_hi - 1), nt - 1);
    const unsigned int bw = (unsigned int)(tx1 - tx0 + 1), last = bw * (unsigned int)(ty1 - ty0 + 1);
    const unsigned int nth = gridDim.x * blockDim.x;
    unsigned int n_all = 0, n_far = 0, n_window = 0, n_occl = 0;
    for(unsigned int k0 = blockIdx.x * blockDim.x; k0 < last; k0 += nth)      // the same trip count CTA-wide
    {
        const unsigned int k = k0 + threadIdx.x;
        bool on = false;
        unsigned int id = 0;
        if(k < last)
        {
            const unsigned int row = k / bw;
            const int ti = tx0 + (int)(k - row * bw), tj = ty0 + (int)row;
            if(max(abs(ti - P.eye_ti), abs(tj - P.eye_tj)) >= ring_lo)
            {
                n_all++;
                const int tc0 = ti * HZ_TILE_CELLS, tr0 = tj * HZ_TILE_CELLS;
                const short2 mt = __ldg(P.mm_tile + (size_t)tj * nt + ti);
                HzBox B;
                const int r = hz_rect_test(P, tc0, min(tc0 + HZ_TILE_CELLS, N - 1), tr0, min(tr0 + HZ_TILE_CELLS, N - 1),
                                           (float)mt.x, (float)mt.y, B);
                if(r == HZ_RECT_DEAD_FAR)         n_far++;
                else if(r == HZ_RECT_DEAD_WINDOW) n_window++;
                else if(r == HZ_RECT_BOXED && hz_box_occluded_thread(P, B, P.occl_tile_max_pix)) n_occl++;
                else { on = true; id = ((unsigned int)tj << 16) | (unsigned int)ti; }
            }
        }
        hz_cta_append(s_app, on, id, P.tile_queue, P.tile_count);
    }
    if(P.stats) hz_cta_stats4(s_stats, P.stats + HZ_STAT_TILES, n_all, n_far, n_window, n_occl);
}

// LOD = false: the reference's mesh (lod = 0 known at compile time: fewer registers, more resident warps); true: the
// instantiation launched once the caller has opted into a coarser far field, P.lod says how coarse this band is
template <bool LOD>
__global__ void __launch_bounds__(256, 3)
k_blocks(const HzView* __restrict__ V)
{
    HZ_KERNEL_PROLOGUE(V, P);
    __shared__ HzCtaAppend s_app;
    __shared__ unsigned int s_stats[4];
    const int nb = P.nb, N = P.N;
    // blocks of (4 << lod) cells: (8 >> lod)^2 of them per tile
    const int lod = LOD ? P.lod : 0, sh = 3 - lod, side = 1 << sh, cells = HZ_BLOCK_CELLS << lod;
    const unsigned int total = *P.tile_count << (2 * sh);
    const unsigned int nth = gridDim.x * blockDim.x;
    unsigned int n_all = 0, n_far = 0, n_window = 0, n_occl = 0;
    for(unsigned int t0 = blockIdx.x * blockDim.x; t0 < total; t0 += nth)     // (the same trip count CTA-wide)
    {
        const unsigned int t = t0 + threadIdx.x;
        bool on = false;
        unsigned int id = 0;
        if(t < total)
        {
            const unsigned int tile = P.tile_queue[t >> (2 * sh)];
            const int tj = (int)(tile >> 16), ti = (int)(tile & 0xFFFFu);
            const int bj = tj * side + (int)((t >> sh) & (unsigned int)(side - 1)), bi = ti * side + (int)(t & (unsigned int)(side - 1));
            if((bj << lod) < nb && (bi << lod) < nb)
            {
                short2 mm = __ldg(P.mm_block + (size_t)(bj << lod) * nb + (bi << lod));
                if(lod > 0)
                {
                    // (min, max) over the 4x4-cell blocks the coarse block is made of
                    int lo = mm.x, hi = mm.y;
                    for(int y = bj << lod; y < min((bj + 1) << lod, nb); y++)
                        for(int x = bi << lod; x < min((bi + 1) << lod, nb); x++)
                        {
                            const short2 c = __ldg(P.mm_block + (size_t)y * nb + x);
                            lo = min(lo, (int)c.x); hi = max(hi, (int)c.y);
                        }
                    mm = make_short2((short)lo, (short)hi);
                }
                HzBox B;
                const int c0 = bi * cells, r0 = bj * cells;
                const int r = hz_rect_test(P, c0, min(c0 + cells, N - 1), r0, min(r0 + cells, N - 1),
                                           (float)mm.x, (float)mm.y, B);
                n_all++;
                if(r == HZ_RECT_DEAD_FAR)         n_far++;
                else if(r == HZ_RECT_DEAD_WINDOW) n_window++;
                else if(r == HZ_RECT_BOXED && hz_box_occluded_thread(P, B, P.occl_block_max_pix)) n_occl++;
                else { on = true; id = ((unsigned int)bj << 16) | (unsigned int)bi; }
            }
        }
        hz_cta_append(s_app, on, id, P.block_queue, P.block_count);
    }
    if(P.stats) hz_cta_stats4(s_stats, P.stats + HZ_STAT_BLOCKS, n_all, n_far, n_window, n_occl);
}

// ---- k_blocks with a level in between (MID) ----------------------------------------------------------------------------
//
// Most of a live tile is dead at the block level (seen at a grazing angle a stretch of terrain is a fraction of a pixel
// high and holds no pixel centre; what does is mostly hidden), and a rectangle test costs a few hundred instructions.
// The MID variant therefore tests the 16 "mids" of every live tile first -- squares of 2x2 blocks = 8x8 cells, (min, max)
// taken from the four blocks' entries of the pyramid -- one per thread, collects the survivors in shared memory, and then
// tests their four blocks each, densely again (thread = (surviving mid, block), 256 at a time): about half the rectangle
// tests per live tile, in full warps.  It is what the views of a batch use (throughput); a lone view is latency-bound
// and keeps the one-level kernel, whose threads have one test each behind them instead of two.
enum { HZ_RECT_OCCLUDED = 4 };

__device__ __forceinline__ int
hz_rect_cull(const HzView& P, int c_lo, int c_hi, int r_lo, int r_hi, float zmin, float zmax, int max_pix)
{
    HzBox B;
    const int r = hz_rect_test(P, c_lo, c_hi, r_lo, r_hi, zmin, zmax, B);
    return (r == HZ_RECT_BOXED && hz_box_occluded_thread(P, B, max_pix)) ? (int)HZ_RECT_OCCLUDED : r;
}

// appends `value` of the threads with `on` to list[*n ...] in shared memory; every thread of the CTA calls, *n was zeroed
// (and the CTA synchronised) before, and the caller synchronises before it reads the list
__device__ __forceinline__ void hz_smem_append(bool on, unsigned int value, unsigned int* list, unsigned int* n)
{
    const unsigned int lane = threadIdx.x & 31u;
    const unsigned int ballot = __ballot_sync(0xffffffffu, on);
    unsigned int base = 0;
    if(lane == 0 && ballot) base = atomicAdd(n, (unsigned int)__popc(ballot));
    base = __shfl_sync(0xffffffffu, base, 0);
    if(on) list[base + __popc(ballot & ((1u << lane) - 1u))] = value;
}

__global__ void __launch_bounds__(256, 3)
k_blocks_mid(const HzView* __restrict__ V)
{
    HZ_KERNEL_PROLOGUE(V, P);
    __shared__ HzCtaAppend s_app;
    __shared__ unsigned int s_mids[256], s_nmids;
    __shared__ unsigned int s_stats[4];
    const int nb = P.nb, N = P.N;
    const int mid_pix = P.occl_tile_max_pix, block_pix = P.occl_block_max_pix;
    const unsigned int total = *P.tile_count * 16u;
    const unsigned int nth = gridDim.x * blockDim.x;
    unsigned int n_all = 0, n_far = 0, n_window = 0, n_occl = 0;
    for(unsigned int t0 = blockIdx.x * blockDim.x; t0 < total; t0 += nth)     // (the same trip counts CTA-wide, here and below)
    {
        __syncthreads();
        if(threadIdx.x == 0) s_nmids = 0;
        __syncthreads();
        {
            const unsigned int t = t0 + threadIdx.x;
            bool on = false;
            unsigned int id = 0;
            if(t < total)
            {
                const unsigned int tile = P.tile_queue[t >> 4];
                const int mj = (int)(tile >> 16) * 4 + (int)((t >> 2) & 3u), mi = (int)(tile & 0xFFFFu) * 4 + (int)(t & 3u);
                const int bj = 2 * mj, bi = 2 * mi;
                if(bj < nb && bi < nb)
                {
                    const short2* mm = P.mm_block + (size_t)bj * nb + bi;
                    const bool right = bi + 1 < nb, up = bj + 1 < nb;
                    const short2 a = __ldg(mm), b = right ? __ldg(mm + 1) : a, c = up ? __ldg(mm + nb) : a,
                                 d = (right && up) ? __ldg(mm + nb + 1) : a;
                    const int lo = min(min((int)a.x, (int)b.x), min((int)c.x, (int)d.x));
                    const int hi = max(max((int)a.y, (int)b.y), max((int)c.y, (int)d.y));
                    const int c0 = bi * HZ_BLOCK_CELLS, r0 = bj * HZ_BLOCK_CELLS;
                    const int r = hz_rect_cull(P, c0, min(c0 + 2 * HZ_BLOCK_CELLS, N - 1), r0, min(r0 + 2 * HZ_BLOCK_CELLS, N - 1),
                                               (float)lo, (float)hi, mid_pix);
                    on = r == HZ_RECT_ALIVE || r == HZ_RECT_BOXED;
                    id = ((unsigned int)mj << 16) | (unsigned int)mi;
                }
            }
            hz_smem_append(on, id, s_mids, &s_nmids);
        }
        __syncthreads();
        const unsigned int items = s_nmids * 4u;
        for(unsigned int jb = 0; jb < items; jb += 256u)
        {
            const unsigned int item = jb + threadIdx.x;
            bool on = false;
            unsigned int id = 0;
            if(item < items)
            {
                const unsigned int mid = s_mids[item >> 2];
                const int bj = (int)(mid >> 16) * 2 + (int)((item >> 1) & 1u), bi = (int)(mid & 0xFFFFu) * 2 + (int)(item & 1u);
                if(bj < nb && bi < nb)
                {
                    const short2 mm = __ldg(P.mm_block + (size_t)bj * nb + bi);
                    const int c0 = bi * HZ_BLOCK_CELLS, r0 = bj * HZ_BLOCK_CELLS;
                    const int r = hz_rect_cull(P, c0, min(c0 + HZ_BLOCK_CELLS, N - 1), r0, min(r0 + HZ_BLOCK_CELLS, N - 1),
                                               (float)mm.x, (float)mm.y, block_pix);
                    n_all++;
                    n_far += (r == HZ_RECT_DEAD_FAR); n_window += (r == HZ_RECT_DEAD_WINDOW); n_occl += (r == HZ_RECT_OCCLUDED);
                    on = r == HZ_RECT_ALIVE || r == HZ_RECT_BOXED;
                    id = ((unsigned int)bj << 16) | (unsigned int)bi;
                }
            }
            hz_cta_append(s_app, on, id, P.block_queue, P.block_count);
        }
    }
    if(P.stats) hz_cta_stats4(s_stats, P.stats + HZ_STAT_BLOCKS, n_all, n_far, n_window, n_occl);
}

__global__ void __launch_bounds__(HZ_WARPS_PER_CTA * 32, HZ_MESH_CTAS)
k_mesh(const HzView* __restrict__ V)
{
    HZ_KERNEL_PROLOGUE(V, P);
    __shared__ HzMeshWarp s_warp[HZ_WARPS_PER_CTA];
    __shared__ unsigned int s_total, s_base;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const HzLaneMap map = hz_lane_map(lane);
    const unsigned int n = *P.block_count;
    const unsigned int nwarps = gridDim.x * HZ_WARPS_PER_CTA;
    // blocks per warp and trip: a full group when there is enough work for that, fewer when warps would otherwise go idle
    const unsigned int per = min((unsigned int)HZ_MESH_GROUP, max(1u, (n + nwarps - 1u) / nwarps));
    unsigned int b = (blockIdx.x * HZ_WARPS_PER_CTA + wib) * per;
    // lane k holds the k-th block of the group
    unsigned int ids = (b + lane < n && lane < per) ? P.block_queue[b + lane] : 0u;
    HzGroupZ Z = {};
    if(b < n) Z = hz_group_heights(P, ids, (int)min(per, n - b), map);
    unsigned int n_meshed = 0, n_tris = 0;
    int count = 0, k_resume = -1;
    HzMeshWarp& M = s_warp[wib];
    while(b < n && k_resume < 0)
    {
        // next group's queue entries and heights first: their latency hides behind this group's arithmetic
        const unsigned int b_next = b + nwarps * per;
        const unsigned int ids_next = (b_next + lane < n && lane < per) ? P.block_queue[b_next + lane] : 0u;
        HzGroupZ Z_next = {};
        if(b_next < n) Z_next = hz_group_heights(P, ids_next, (int)min(per, n - b_next), map);
        const int nblk = (int)min(per, n - b);
        hz_group_project(P, ids, nblk, lane, map, Z, M);
        k_resume = hz_group_triangles<false>(P, ids, 0, nblk, lane, M, count, n_tris);
        __syncwarp();
        n_meshed += (unsigned int)nblk;
        if(k_resume < 0) { b = b_next; ids = ids_next; Z = Z_next; }
    }
    if(k_resume >= 0)
    {
        // the triangle list is full: this warp draws everything else it finds itself (b, ids: the group it stopped in,
        // already projected).  Out of line, with its own registers: see hz_mesh_slow_tail.
        hz_mesh_slow_tail(P, M, count, b, n, nwarps * per, (int)per, ids, k_resume, nullptr, n_meshed, n_tris);
        count = 0;
    }
    hz_stage_flush_cta(P, s_warp[wib], count, &s_total, &s_base);
    if(P.stats && lane == 0 && n_meshed)
    {
        atomicAdd(P.stats + HZ_STAT_BLOCKS_MESHED, n_meshed);
        atomicAdd(P.stats + HZ_STAT_TRIANGLES, n_tris);
    }
}

// ---- the triangles the lanes of a warp draw themselves (bounding boxes of a few dozen pixels at most) -----------------
//
// Coverage and shading are separated here as in k_big: every lane walks the bounding box of ITS triangle one pixel
// centre per step, stepping 32-bit edge functions, and the covered ones of all lanes are compacted into a small list in
// shared memory (owner lane, offset in the box); whenever the list holds 32 the lanes shade 32 fragments at once, each
// fetching its fragment's plane equations from the owner's row of a table in shared memory.  Walking and shading in
// the same loop instead leaves most lanes idle through the ~45 instructions of every fragment: a triangle covers a few
// of the pixel centres of its box, and every lane's are somewhere else.
struct HzFragAttr          // what hz_fragment needs of a triangle; one row per lane, 16 words
{
    float xw0, yw0, z0w, dzdx, dzdy, zw_lo, zw_hi, r0, drdx, drdy;
    unsigned int id;
    int px0, py0;
    int pad[3];
};
struct HzRasterWarp
{
    HzFragAttr   attr[32];
    unsigned int frag[64];         // owner | dx << 5 | dy << 11
};

__device__ __forceinline__ void hz_shade_listed(const HzView& P, const HzRasterWarp& S, unsigned int entry)
{
    const HzFragAttr& A = S.attr[entry & 31u];
    HzTri T;                       // (only the members hz_fragment reads)
    T.xw0 = A.xw0; T.yw0 = A.yw0; T.z0w = A.z0w; T.dzdx = A.dzdx; T.dzdy = A.dzdy; T.zw_lo = A.zw_lo; T.zw_hi = A.zw_hi;
    T.r0 = A.r0; T.drdx = A.drdx; T.drdy = A.drdy; T.id = A.id;
    hz_fragment(P, T, A.px0 + (int)((entry >> 5) & 63u), A.py0 + (int)(entry >> 11));
}

// All lanes of the warp call; `mine`: this lane has a set-up triangle T to draw (its box at most 64 x 64 pixels and
// hz_tri_is_small).
__device__ __forceinline__ void hz_draw_boxes_warp(const HzView& P, const HzTri& T, bool mine, HzRasterWarp& S, unsigned int lane)
{
    const unsigned int any = __ballot_sync(0xffffffffu, mine);
    if(any == 0) return;
    int bw = 0, npx = 0;
    int e0 = 0, e1 = 0, e2 = 0, sx0 = 0, sx1 = 0, sx2 = 0, wr0 = 0, wr1 = 0, wr2 = 0;
    if(mine)
    {
        HzFragAttr& A = S.attr[lane];
        A.xw0 = T.xw0; A.yw0 = T.yw0; A.z0w = T.z0w; A.dzdx = T.dzdx; A.dzdy = T.dzdy; A.zw_lo = T.zw_lo; A.zw_hi = T.zw_hi;
        A.r0 = T.r0; A.drdx = T.drdx; A.drdy = T.drdy; A.id = T.id; A.px0 = T.px0; A.py0 = T.py0;
        const HzEdges<int> E(T);
        const int Px = T.px0 * 256 + 128, Py = T.py0 * 256 + 128;
        e0 = E.dx0 * (Py - T.Y0) - E.dy0 * (Px - T.X0) - E.b0;      // >= 0 <=> inside, per edge
        e1 = E.dx1 * (Py - T.Y1) - E.dy1 * (Px - T.X1) - E.b1;
        e2 = E.dx2 * (Py - T.Y2) - E.dy2 * (Px - T.X2) - E.b2;
        bw = T.px1 - T.px0 + 1;
        npx = bw * (T.py1 - T.py0 + 1);
        sx0 = E.dy0 * 256; sx1 = E.dy1 * 256; sx2 = E.dy2 * 256;   // one pixel to the right: E -= dy * 256
        wr0 = E.dx0 * 256 + bw * sx0; wr1 = E.dx1 * 256 + bw * sx1; wr2 = E.dx2 * 256 + bw * sx2;   // up a row and back to its left end
    }
    const int steps = __reduce_max_sync(0xffffffffu, npx);
    const unsigned int below = (1u << lane) - 1u;
    unsigned int count = 0;        // entries in the list (the same in all lanes)
    int x = 0, y = 0;
    __syncwarp();
    for(int s = 0; s < steps; s++)
    {
        const bool in = s < npx && (e0 | e1 | e2) >= 0;
        const unsigned int m = __ballot_sync(0xffffffffu, in);
        if(in) S.frag[count + __popc(m & below)] = lane | ((unsigned int)x << 5) | ((unsigned int)y << 11);
        count += __popc(m);
        e0 -= sx0; e1 -= sx1; e2 -= sx2;
        if(++x == bw) { x = 0; y++; e0 += wr0; e1 += wr1; e2 += wr2; }
        if(count >= 32u)
        {
            __syncwarp();
            hz_shade_listed(P, S, S.frag[lane]);
            const unsigned int rest = (lane < count - 32u) ? S.frag[32u + lane] : 0u;
            __syncwarp();
            if(lane < count - 32u) S.frag[lane] = rest;
            count -= 32u;
        }
    }
    __syncwarp();
    if(lane < count) hz_shade_listed(P, S, S.frag[lane]);
    __syncwarp();                  // the table and the list are free for the next trip
}

// ---- k_raster: one thread per triangle of a stage's list

#ifndef HZ_RASTER_CTAS
#define HZ_RASTER_CTAS 3           /* resident CTAs per SM k_raster is compiled for (register budget 80; measured: 2 CTAs, 108 */
                                   /* registers and no spills, 3-4 % slower; 4 CTAs, 64 registers, +1.5 % in batches, lone views 1 % slower) */
#endif
__global__ void __launch_bounds__(256, HZ_RASTER_CTAS)
k_raster(const HzView* __restrict__ V)
{
    HZ_KERNEL_PROLOGUE(V, P);
    __shared__ HzRasterWarp s_warp[8];
    const unsigned int n = min(*P.tri_count, P.tri_capacity);
    const unsigned int nth = gridDim.x * blockDim.x;
    const unsigned int lane = threadIdx.x & 31u;
    unsigned int n_big = 0;
    for(unsigned int t0 = blockIdx.x * blockDim.x + threadIdx.x - lane; t0 < n; t0 += nth)    // warp-uniform trips
    {
        const unsigned int t = t0 + lane;
        HzTri T;
        unsigned int id = 0, nx = 0, k = 0, nsub = 0;
        int st = HZ_SETUP_NOTHING;
        if(t < n)
        {
            id = P.tri_queue[t];
            st = hz_tri_setup(P, id, 0, T);
            if(st == HZ_SETUP_OK) nsub = hz_big_layout(P, T, nx, k);
        }
        // Who draws what: bounding boxes up to P.small_max_pix pixels are drawn here.  Middle-sized ones (up to
        // P.mid_max_pix) too where many lanes of the warp have one -- zoomed-in views, where neighbouring triangles are
        // all that size; for a few of them a warp of its own in k_big is the better deal.  Everything else is queued.
        bool mine = (st == HZ_SETUP_OK && nsub == 0);
        {
            const bool mid = st == HZ_SETUP_OK && nsub != 0 && (T.px1 - T.px0 + 1) * (T.py1 - T.py0 + 1) <= P.mid_max_pix &&
                             hz_tri_is_small(T) && T.px1 - T.px0 < 64 && T.py1 - T.py0 < 64;
            if(__popc(__ballot_sync(0xffffffffu, mid)) >= HZ_MID_LANES && mid) { mine = true; nsub = 0; }
        }
        hz_draw_boxes_warp(P, T, mine, s_warp[threadIdx.x >> 5], lane);
        // the large ones of the warp reserve their queue slots and records with ONE atomic each: in a zoomed-in view
        // nearly every triangle is large, and a million same-address atomics would be the whole kernel
        const unsigned int ballot = __ballot_sync(0xffffffffu, nsub != 0);
        if(ballot)
        {
            unsigned int incl = nsub;
            #pragma unroll
            for(int d = 1; d < 32; d <<= 1)
            {
                const unsigned int up = __shfl_up_sync(0xffffffffu, incl, d);
                if((int)lane >= d) incl += up;
            }
            const unsigned int total = __shfl_sync(0xffffffffu, incl, 31);
            unsigned int slot0 = 0, rec0 = 0;
            if(lane == 0) { slot0 = atomicAdd(P.big_count, total); rec0 = atomicAdd(P.bigtri_count, (unsigned int)__popc(ballot)); }
            slot0 = __shfl_sync(0xffffffffu, slot0, 0); rec0 = __shfl_sync(0xffffffffu, rec0, 0);
            if(nsub != 0)
            {
                if(hz_big_enqueue(P, T, id, 0, nx, k, nsub, slot0 + incl - nsub, rec0 + __popc(ballot & ((1u << lane) - 1u))))
                    n_big += nsub;
                else
                    st = HZ_SETUP_QUEUE_FULL;
            }
        }
        // the rare cases, out of line and only here, where nothing of the triangle's set-up is live any more: the queue
        // was full (never on the normal path) or the triangle straddles the seam (opt-in seam wrap)
        if(st < 0) n_big += hz_raster_rare(P, id, st);
    }
    n_big = hz_warp_sum(n_big);
    if(P.stats && lane == 0 && n_big) atomicAdd(P.stats + HZ_STAT_BIG_ENTRIES, n_big);
}

cudaError_t hz_launch_raster(const HzView& v, const HzView* d_v, int nviews, cudaStream_t stream)
{
    return hz_launch(k_raster, dim3(hz_grid(v, 6, nviews), (unsigned)nviews), dim3(256), stream, d_v);
}

// `worst_case`: size the tile kernel for any eye position (a CUDA graph is captured once per context and replayed
// for every view); otherwise for this view's eye tile, and nothing is launched if the band is empty.
cudaError_t hz_launch_band(const HzView& v, const HzView* d_v, int nviews, bool worst_case, cudaStream_t stream, int* launches)
{
    *launches = 0;
    const int rmax = worst_case ? v.nt - 1
                                : max(max(v.eye_ti, v.nt - 1 - v.eye_ti), max(v.eye_tj, v.nt - 1 - v.eye_tj));
    // (With the opt-in level of detail the bands' limits depend on each view's azimuth window: a launch that serves
    // several views, or a captured graph that will be replayed for others, must not be shaped by this one's.)
    const bool any_band = worst_case && v.lod_capable;
    const int ring_hi = any_band ? v.nt : min(v.ring_hi, rmax + 1);
    if(!any_band && v.ring_lo >= ring_hi) return cudaSuccess;
    // (the threads walk the band's bounding square, clipped to the mesh)
    const long long side = min(2 * ring_hi - 1, v.nt), ntiles = side * side;
    long long ctas = (ntiles + 255) / 256;
    if(ctas > (long long)hz_grid(v, 8, nviews)) ctas = hz_grid(v, 8, nviews);
    const unsigned int ny = (unsigned int)nviews;
    cudaError_t e;
    void (*blocks)(const HzView*) = v.lod_capable ? k_blocks<true> : (v.mid_level ? k_blocks_mid : k_blocks<false>);
    if((e = hz_launch(k_tiles, dim3((unsigned)ctas, ny), dim3(256), stream, d_v)) != cudaSuccess) return e;
    if((e = hz_launch(blocks,  dim3(hz_grid(v, 8, nviews), ny), dim3(256), stream, d_v)) != cudaSuccess) return e;
    *launches = 4;
    if((e = hz_launch(k_mesh,   dim3(hz_grid(v, 4, nviews), ny), dim3(HZ_WARPS_PER_CTA * 32), stream, d_v)) != cudaSuccess) return e;
    if((e = hz_launch(k_raster, dim3(hz_grid(v, 6, nviews), ny), dim3(256), stream, d_v)) != cudaSuccess) return e;
    return cudaSuccess;
}

// ================================================================================================
// k_big: one warp per (triangle, sub-box), lanes spread over the sub-box's pixels
// ================================================================================================

// Coverage and shading are separated: lane = column of the sub-box steps its edge functions down the rows, four rows
// at a time, and the covered pixel centres of those four rows are compacted through shared memory (`slots`, 128 bytes
// per warp); then the lanes shade them densely, 32 at a time.  (Shading where the coverage test ran would leave most
// lanes idle through the ~45 instructions of a fragment: a triangle covers a few pixels of each row of its sub-box.)
// The whole warp calls, with the same arguments but for `lane`.
template <typename I>
__device__ __forceinline__ void
hz_draw_subbox(const HzView& P, const HzTri& T, int x0, int x1, int y0, int y1, int lane, uint8_t* slots)
{
    const HzEdges<I> E(T);
    if(E.box_outside(T, x0, x1, y0, y1)) return;
    const int px = x0 + lane;
    const bool column = px <= x1;
    const I Px = (I)px * 256 + 128, Py = (I)y0 * 256 + 128;
    I e0 = E.dx0 * (Py - T.Y0) - E.dy0 * (Px - T.X0) - E.b0;      // >= 0 <=> inside, per edge
    I e1 = E.dx1 * (Py - T.Y1) - E.dy1 * (Px - T.X1) - E.b1;
    I e2 = E.dx2 * (Py - T.Y2) - E.dy2 * (Px - T.X2) - E.b2;
    const I sy0 = E.dx0 * 256, sy1 = E.dx1 * 256, sy2 = E.dx2 * 256;
    const unsigned int below = (1u << lane) - 1u;
    for(int yb = y0; yb <= y1; yb += 4)
    {
        unsigned int n = 0;                                       // covered pixel centres of these rows (the same in all lanes)
        #pragma unroll
        for(int r = 0; r < 4; r++)
        {
            const bool in = column && yb + r <= y1 && (e0 | e1 | e2) >= 0;
            const unsigned int m = __ballot_sync(0xffffffffu, in);
            if(in) slots[n + __popc(m & below)] = (uint8_t)((r << 5) | lane);
            n += __popc(m);
            e0 += sy0; e1 += sy1; e2 += sy2;
        }
        if(n == 0) continue;
        __syncwarp();
        for(unsigned int f = lane; f < n; f += 32)
        {
            const unsigned int code = slots[f];
            hz_fragment(P, T, x0 + (int)(code & 31u), yb + (int)(code >> 5));
        }
        __syncwarp();
    }
}

#ifndef HZ_BIG_CTAS
#define HZ_BIG_CTAS 4              /* resident CTAs per SM k_big is compiled for: 64 registers (left to itself ptxas takes 72, */
                                   /* 3 CTAs: measured 2 % slower in batches, 4 % in the 5-degree zoom) */
#endif
__global__ void __launch_bounds__(256, HZ_BIG_CTAS)
k_big(const HzView* __restrict__ V)
{
    HZ_KERNEL_PROLOGUE(V, P);
    // every slot below min(count, capacity) was written: with a record index or a triangle number, or poisoned by a
    // triangle that found the queue exhausted and drew itself (hz_raster_one)
    __shared__ uint8_t s_slots[8][128];
    unsigned int count = *P.big_count;
    if(count > P.big_capacity) count = P.big_capacity;
    const int lane = threadIdx.x & 31;
    uint8_t* slots = s_slots[threadIdx.x >> 5];
    const unsigned int nwarps = gridDim.x * (blockDim.x >> 5);
    for(unsigned int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < count; t += nwarps)
    {
        const uint2 entry = __ldcg(P.big_queue + t);
        if(entry.x == 0xFFFFFFFFu) continue;                                   // poisoned slot
        HzTri T;
        if(entry.y & HZ_BIG_RECOMPUTE)
        {
            if(hz_tri_setup(P, entry.x, (int)((entry.y >> 28) & 3u), T) != HZ_SETUP_OK) continue;   // cannot happen
        }
        else hz_tri_load(P.bigtri + (size_t)entry.x * HZ_TRI_RECORD_VEC, T);
        const int rows = HZ_BIG_ROWS << ((entry.y >> 24) & 15u);
        const int y0 = T.py0 + (int)(entry.y & 0xFFFu) * rows,                y1 = min(y0 + rows - 1, T.py1);
        const int x0 = T.px0 + (int)((entry.y >> 12) & 0xFFFu) * HZ_BIG_COLS, x1 = min(x0 + HZ_BIG_COLS - 1, T.px1);
        if(hz_tri_is_small(T)) hz_draw_subbox<int>(P, T, x0, x1, y0, y1, lane, slots);
        else                   hz_draw_subbox<long long>(P, T, x0, x1, y0, y1, lane, slots);
    }
}

cudaError_t hz_launch_big(const HzView& v, const HzView* d_v, int nviews, cudaStream_t stream)
{
    return hz_launch(k_big, dim3(hz_grid(v, 8, nviews), (unsigned)nviews), dim3(256), stream, d_v);
}

// ================================================================================================
// k_resolve
// ================================================================================================

// lib:1013-1025 for one pixel: depth as glReadPixels(GL_DEPTH_COMPONENT, GL_FLOAT) returns it -> range
__device__ __forceinline__ float hz_range_of_q(unsigned int q, float tanel, float znear, float zfar)
{
    // lib:1016 "depth == 1.0f -> -1": of the 24-bit values only the cleared one reads back as 1.0f (the next lower
    // one is 1 - 2^-24, exactly representable).  Checked first: most of a panorama is sky, and the rest of this
    // function is FP64.
    if(q == HZ_Q_MAX) return -1.0f;
    const float depth = (float)((double)q * (1.0 / 16777215.0));             // F7 read-back
    const float length_en = depth * (zfar - znear) + znear;                  // lib:1018
    const float z = tanel * length_en;
    // hypotf (lib:1024): glibc evaluates it in double and rounds once
    return (float)sqrt((double)length_en * (double)length_en + (double)z * (double)z);
}

// Where k_resolve writes.  Normally one destination that is exactly the target (columns [x0,x1), row stride
// x1-x0).  For a panorama split by azimuth wedge over several GPUs the destinations are the FULL panoramas of every
// rank (peer memory, written over NVLink): row stride W, this wedge's columns at offset x0 -- the gather of the
// shards is fused into the kernel that produces them.
struct HzResolve
{
    const unsigned long long* vis;
    int   Wt, H;                 // target width (x1-x0), height
    const float* tanel;          // [H] tan(elevation) per GL row, host-computed (lib:1007-1012)
    float znear, zfar;
    int   n_out, out_stride, out_x0;
};

__device__ __forceinline__ HzResolve hz_resolve_params(const HzView& P)
{
    HzResolve R;
    R.vis = P.vis; R.Wt = P.x1 - P.x0; R.H = P.H; R.tanel = P.tanel; R.znear = P.znear; R.zfar = P.zfar;
    R.n_out = P.n_out; R.out_stride = P.out_stride; R.out_x0 = P.out_x0;
    return R;
}

// 4 pixels per thread and trip: 2x16 B of keys in, 12 B of BGR and 16 B of range out (per destination).  A CTA works on
// one row of the target: no index arithmetic to speak of (the first version spent more instructions on finding its
// row, a division, than on its four pixels), the row's tan(elevation) is read once, and the next trip's keys are on
// their way while this trip's pixels are converted.  Two launch shapes: for several views one CTA per row (grid x = row),
// whose threads take a few trips each -- fewest instructions; for a lone view, which is latency-bound and whose
// terrain pixels each cost a double-precision square root, the row is spread over as many CTAs as it has groups of
// 256 (grid x = part of the row, grid z = row): one trip per thread.
__global__ void __launch_bounds__(HZ_CTA_THREADS)
k_resolve4(const HzView* __restrict__ V)
{
    HZ_KERNEL_PROLOGUE(V, P);
    const unsigned int Wt = (unsigned int)(P.x1 - P.x0), gpr = Wt >> 2;        // groups of 4 pixels per row
    const bool spread = gridDim.z > 1;
    const unsigned int y = spread ? blockIdx.z : blockIdx.x;                    // GL row (0 = bottom)
    const unsigned int stride = spread ? HZ_CTA_THREADS * gridDim.x : HZ_CTA_THREADS;
    const unsigned int ep = P.epoch;
    const float znear = P.znear, zfar = P.zfar;
    const int n_out = P.n_out;
    uint8_t* const image0 = P.out_image[0];
    float* const ranges0 = P.out_ranges[0];
    const float tanel = ranges0 != nullptr ? __ldg(P.tanel + y) : 0.0f;
    const ulonglong2* src = (const ulonglong2*)(P.vis + (size_t)y * Wt);
    const size_t dst_row = (size_t)((unsigned int)P.H - 1u - y) * (unsigned int)P.out_stride + (unsigned int)P.out_x0;   // top row first (lib:949-958, 1026-1038)

    unsigned int xg = threadIdx.x + (spread ? HZ_CTA_THREADS * blockIdx.x : 0u);
    ulonglong2 k01 = make_ulonglong2(0, 0), k23 = k01;
    if(xg < gpr) { k01 = __ldcs(src + 2 * xg); k23 = __ldcs(src + 2 * xg + 1); }   // read once: streaming
    while(xg < gpr)
    {
        const unsigned int xg_next = xg + stride;
        ulonglong2 n01 = k01, n23 = k23;
        if(xg_next < gpr) { n01 = __ldcs(src + 2 * xg_next); n23 = __ldcs(src + 2 * xg_next + 1); }

        const unsigned int q0 = hz_key_q(k01.x, ep), q1 = hz_key_q(k01.y, ep), q2 = hz_key_q(k23.x, ep), q3 = hz_key_q(k23.y, ep);
        // hit: (B,G,R) = (0,0,r8) ; sky: clear colour (0,0,1) read as BGR = (255,0,0)   lib:185, 938-939
        // bytes B0 G0 R0 B1 | G1 R1 B2 G2 | R2 B3 G3 R3
        const unsigned int B0 = q0 != HZ_Q_MAX ? 0u : 255u, R0 = q0 != HZ_Q_MAX ? (unsigned int)k01.x & 0xFFu : 0u;
        const unsigned int B1 = q1 != HZ_Q_MAX ? 0u : 255u, R1 = q1 != HZ_Q_MAX ? (unsigned int)k01.y & 0xFFu : 0u;
        const unsigned int B2 = q2 != HZ_Q_MAX ? 0u : 255u, R2 = q2 != HZ_Q_MAX ? (unsigned int)k23.x & 0xFFu : 0u;
        const unsigned int B3 = q3 != HZ_Q_MAX ? 0u : 255u, R3 = q3 != HZ_Q_MAX ? (unsigned int)k23.y & 0xFFu : 0u;
        const uint32_t w0 = B0 | (R0 << 16) | (B1 << 24);
        const uint32_t w1 = (R1 << 8) | (B2 << 16);
        const uint32_t w2 = R2 | (B3 << 8) | (R3 << 24);

        float4 r = make_float4(-1.0f, -1.0f, -1.0f, -1.0f);
        // most groups of four pixels are sky: skip the FP64 conversion for them altogether
        if(ranges0 != nullptr && (q0 & q1 & q2 & q3) != HZ_Q_MAX)
        {
            r.x = hz_range_of_q(q0, tanel, znear, zfar);
            r.y = hz_range_of_q(q1, tanel, znear, zfar);
            r.z = hz_range_of_q(q2, tanel, znear, zfar);
            r.w = hz_range_of_q(q3, tanel, znear, zfar);
        }
        const size_t dst = dst_row + 4u * xg;
        if(image0)
        {
            uint32_t* o = (uint32_t*)(image0 + dst * 3);       // dst*3 is a multiple of 4 because x, x0 and the stride are
            o[0] = w0; o[1] = w1; o[2] = w2;
        }
        if(ranges0) *(float4*)(ranges0 + dst) = r;
        for(int d = 1; d < n_out; d++)                         // (the other ranks of a wedge-sharded panorama)
        {
            uint8_t* image = P.out_image[d];
            float* ranges = P.out_ranges[d];
            if(image)
            {
                uint32_t* o = (uint32_t*)(image + dst * 3);
                o[0] = w0; o[1] = w1; o[2] = w2;
            }
            if(ranges) *(float4*)(ranges + dst) = r;
        }
        xg = xg_next; k01 = n01; k23 = n23;
    }
}

// any width
__global__ void __launch_bounds__(256)
k_resolve1(const HzView* __restrict__ V)
{
    HZ_KERNEL_PROLOGUE(V, P);
    const HzResolve R = hz_resolve_params(P);
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if(g >= (long long)R.Wt * R.H) return;
    const int y = (int)(g / R.Wt), x = (int)(g % R.Wt);
    const unsigned long long key = R.vis[g];
    const size_t dst = (size_t)(R.H - 1 - y) * R.out_stride + R.out_x0 + x;
    const unsigned int q = hz_key_q(key, P.epoch);
    const bool hit = q != HZ_Q_MAX;
    const float range = (P.out_ranges[0] != nullptr) ? hz_range_of_q(q, R.tanel[y], R.znear, R.zfar) : -1.0f;
    for(int d = 0; d < R.n_out; d++)
    {
        uint8_t* image = P.out_image[d];
        float* ranges = P.out_ranges[d];
        if(image)
        {
            image[dst * 3 + 0] = hit ? 0 : 255;
            image[dst * 3 + 1] = 0;
            image[dst * 3 + 2] = hit ? (unsigned char)(key & 0xFFu) : 0;
        }
        if(ranges) ranges[dst] = range;
    }
}

bool hz_resolve_is_vectorisable(const HzView& v)
{
    if((v.x1 - v.x0) % 4 != 0 || v.out_stride % 4 != 0 || v.out_x0 % 4 != 0) return false;
    for(int d = 0; d < v.n_out; d++)
        if(((uintptr_t)v.out_image[d] & 3) != 0 || ((uintptr_t)v.out_ranges[d] & 15) != 0) return false;
    return true;
}

// every view of one launch must pass the same hz_resolve_is_vectorisable() (the caller checks)
cudaError_t hz_launch_resolve(const HzView& v, const HzView* d_v, int nviews, cudaStream_t stream)
{
    const int Wt = v.x1 - v.x0;
    if(hz_resolve_is_vectorisable(v))
    {
        const unsigned int parts = (unsigned)((Wt / 4 + HZ_CTA_THREADS - 1) / HZ_CTA_THREADS);
        if(nviews == 1 && v.H > 1 && v.H <= 65535)
            return hz_launch(k_resolve4, dim3(parts, 1u, (unsigned)v.H), dim3(HZ_CTA_THREADS), stream, d_v);
        return hz_launch(k_resolve4, dim3((unsigned)v.H, (unsigned)nviews), dim3(HZ_CTA_THREADS), stream, d_v);
    }
    else
    {
        const long long n = (long long)Wt * v.H;
        return hz_launch(k_resolve1, dim3((unsigned)((n + 255) / 256), (unsigned)nviews), dim3(256), stream, d_v);
    }
}

// ================================================================================================
// k_peer_barrier: barrier between the ranks of a wedge-sharded panorama, on the GPUs, through peer memory
// ================================================================================================
//
// Every rank owns an array arrive[HZ_MAX_OUT] (+ one error word) that its peers have mapped.  Rank i announces epoch e
// by storing e into arrive[i] of every rank (release, system scope: everything this stream did before, e.g. the
// resolve kernel's peer stores, is visible first), then waits until all entries of its own array have reached e.
// The wait is bounded: a rank that never arrives must not hang the others' GPUs; a timeout is recorded in the
// error word (the caller checks it) and the kernel returns.
__global__ void __launch_bounds__(32)
k_peer_barrier(HzPeerFlags F, unsigned int epoch)
{
    const unsigned int r = threadIdx.x;
    if(r >= (unsigned int)F.n) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(F.arrive[r] + F.rank), "r"(epoch) : "memory");
    unsigned int seen = 0;
    for(unsigned int spin = 0; spin < (1u << 20); spin++)
    {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(F.arrive[F.rank] + r) : "memory");
        if((int)(seen - epoch) >= 0) return;
        __nanosleep(64);
    }
    atomicAdd(F.arrive[F.rank] + HZ_MAX_OUT, 1u);            // timed out
}

cudaError_t hz_launch_peer_barrier(const HzPeerFlags& f, unsigned int epoch, cudaStream_t stream)
{
    k_peer_barrier<<<1, 32, 0, stream>>>(f, epoch);
    return cudaGetLastError();
}

// ================================================================================================
// k_horizon: per image column, the topmost terrain pixel (row, range); -1 / -1.0f if the column is all sky
// ================================================================================================

__global__ void __launch_bounds__(256)
k_horizon(const float* __restrict__ ranges, int n, int W, int H, int* __restrict__ rows, float* __restrict__ range)
{
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if(g >= (long long)n * W) return;
    const int img = (int)(g / W), x = (int)(g % W);
    const float* col = ranges + (size_t)img * W * H + x;
    int row = -1; float r = -1.0f;
    for(int y = 0; y < H; y++)
    {
        const float v = col[(size_t)y * W];
        if(v > 0.0f) { row = y; r = v; break; }
    }
    rows[g] = row; range[g] = r;
}

cudaError_t hz_launch_horizon(const float* ranges, int n, int W, int H, int* rows, float* range, cudaStream_t stream)
{
    const long long total = (long long)n * W;
    if(total <= 0) return cudaSuccess;
    k_horizon<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(ranges, n, W, H, rows, range);
    return cudaGetLastError();
}

// ================================================================================================
// k_viewshed: R2 ray casting (include/horizonator-batch.h states the definition; oracle/viewshed_oracle.c restates it
// operation for operation, and the masks must agree bit for bit).  Every operation of a ray is written as an
// explicitly rounded intrinsic, so that neither -fmad nor the optimiser can contract or reorder it.
// ================================================================================================

// metres from the eye along one axis at cell coordinate x (vertex.glsl:128-130 with x in place of the vertex index, as
// k_prepare's axis tables): scale = cos_viewer_lat east, 1 north
__device__ __forceinline__ float hz_vs_metres(float x, float v, float dpc, float scale)
{
    return __fmul_rn(__fdiv_rn(__fmul_rn(__fmul_rn(__fmul_rn(__fsub_rn(x, v), dpc), HZ_REARTH_F), HZ_PI_F), 180.f), scale);
}

// A lane collects the bits of one mask word while its ray stays inside that word (a column-stepping ray crosses a new
// word every 32 steps or when its row changes) and hands them on when it leaves it; lanes handing on the same word
// merge their bits first (a row-stepping warp's 32 rays usually land in one or two words), so one atomicOr per word.
// Warp-collective: every lane of the warp calls it at the same step.
__device__ __forceinline__ void hz_vs_collect(uint32_t*& pend, uint32_t& pbits, uint32_t* word, uint32_t bit, bool last,
                                              unsigned int lane)
{
    const bool change = word != nullptr && word != pend;
    const bool flush = pbits != 0u && (change || last);
    const unsigned int fm = __ballot_sync(0xffffffffu, flush);
    if(flush)
    {
        const unsigned int peers = __match_any_sync(fm, (unsigned long long)pend);
        const unsigned int v = __reduce_or_sync(peers, pbits);
        if(lane == (unsigned int)(__ffs(peers) - 1)) atomicOr(pend, v);
    }
    if(change) { pend = word; pbits = bit; }
    else pbits = last ? 0u : (pbits | bit);
}

#define HZ_VS_WARPS  4     /* warps per CTA */
#define HZ_VS_UNROLL 4     /* steps whose heights are loaded before the first of them is evaluated */

// One thread per ray, gridDim.y = view.  The 4N-4 rays go to warps side by side: bottom row, top row, left column,
// right column (without the corners), each side padded to whole warps, so that a warp holds 32 adjacent rays.  A
// warp's rays run for a common number of steps (each lane's own count masks the rest): a side's rays that step
// along the same axis all end on the same column or row, and the collective hand-on of mask bits needs every lane.
__global__ void __launch_bounds__(HZ_VS_WARPS * 32)
k_viewshed(const __grid_constant__ HzViewshed p)
{
    const int N = p.N;
    const HzViewshedEye E = p.eye[blockIdx.y];
    uint32_t* const mask = p.masks + (size_t)blockIdx.y * N * p.w32;
    if(blockIdx.x == 0 && threadIdx.x < 4)
    {
        // the four vertices around the eye
        const int i = (int)floorf(E.vci) + (int)(threadIdx.x & 1), j = (int)floorf(E.vcj) + (int)(threadIdx.x >> 1);
        atomicOr(mask + (size_t)j * p.w32 + (i >> 5), 1u << (i & 31));
    }

    const unsigned int lane = threadIdx.x & 31;
    int w = (int)(blockIdx.x * HZ_VS_WARPS + (threadIdx.x >> 5));
    const int wrow = (N + 31) >> 5, wcol = (N - 2 + 31) >> 5;
    int ti, tj;
    bool valid;
    if(w < 2 * wrow)
    {
        const int k = (w % wrow) * 32 + (int)lane;
        valid = k < N; ti = k; tj = w < wrow ? 0 : N - 1;
    }
    else
    {
        w -= 2 * wrow;
        if(w >= 2 * wcol) return;                             // whole warps only
        const int k = (w % wcol) * 32 + (int)lane;
        valid = k < N - 2; ti = w < wcol ? 0 : N - 1; tj = k + 1;
    }

    // "a" is the axis the ray steps along, "b" the other one
    const float di = __fsub_rn((float)ti, E.vci), dj = __fsub_rn((float)tj, E.vcj);
    const bool xmaj = fabsf(di) >= fabsf(dj);
    const float va = xmaj ? E.vci : E.vcj, vb = xmaj ? E.vcj : E.vci;
    const float da = xmaj ? di : dj, db = xmaj ? dj : di;
    const float sa = xmaj ? E.cos_lat : 1.0f, sb = xmaj ? 1.0f : E.cos_lat;
    const int ta = xmaj ? ti : tj;
    const float slope = da != 0.f ? __fdiv_rn(db, da) : 0.f;
    const int step = da > 0.f ? 1 : -1;
    const int a0 = da > 0.f ? (int)floorf(va) + 1 : (int)ceilf(va) - 1;
    const int nsteps = (valid && da != 0.f) ? abs(ta - a0) + 1 : 0;
    const int maxsteps = (int)__reduce_max_sync(0xffffffffu, (unsigned int)nsteps);

    // height at (a, b): mosaic[b][a] on a column-stepping ray (its warp reads 32 rows of one column per step; a
    // transposed copy of the mosaic for these rays measured 3 % slower, DESIGN.md section 9), mosaic[a][b] on a
    // row-stepping one
    const int16_t* const base = p.mosaic;
    const size_t stride_a = xmaj ? 1 : (size_t)p.pitch, stride_b = xmaj ? (size_t)p.pitch : 1;
    const float vz = E.vz, curv = p.curvature, th = p.target_height, dpc = p.deg_per_cell;

    float smax = __int_as_float(0xff800000);                  // -inf
    uint32_t* pend = nullptr;
    uint32_t pbits = 0;
    for(int k0 = 0; k0 < maxsteps; k0 += HZ_VS_UNROLL)
    {
        // the addresses of the next steps do not depend on the running maximum: their loads go out first
        float zlo[HZ_VS_UNROLL], zhi[HZ_VS_UNROLL];
        #pragma unroll
        for(int u = 0; u < HZ_VS_UNROLL; u++)
        {
            zlo[u] = zhi[u] = 0.f;
            if(k0 + u < nsteps)
            {
                const int a = a0 + (k0 + u) * step;
                const float b = __fadd_rn(vb, __fmul_rn(__fsub_rn((float)a, va), slope));
                const int b0 = min(max((int)floorf(b), 0), N - 2);
                const int16_t* q = base + (size_t)a * stride_a + (size_t)b0 * stride_b;
                zlo[u] = (float)__ldg(q);
                zhi[u] = (float)__ldg(q + stride_b);
            }
        }
        #pragma unroll
        for(int u = 0; u < HZ_VS_UNROLL; u++)
        {
            uint32_t* word = nullptr;
            uint32_t bit = 0;
            if(k0 + u < nsteps)
            {
                const int a = a0 + (k0 + u) * step;
                const float b = __fadd_rn(vb, __fmul_rn(__fsub_rn((float)a, va), slope));
                const int b0 = min(max((int)floorf(b), 0), N - 2);
                const int r = min(max(__float2int_rn(b), 0), N - 1);
                // the surface at (a, b): linear along the grid edge between b0 and b0 + 1
                const float t = __fsub_rn(b, (float)b0);
                const float z = __fadd_rn(zlo[u], __fmul_rn(__fsub_rn(zhi[u], zlo[u]), t));
                const float ma = hz_vs_metres((float)a, va, dpc, sa), mb = hz_vs_metres(b, vb, dpc, sb);
                const float d2 = __fadd_rn(__fmul_rn(ma, ma), __fmul_rn(mb, mb));
                const float s = __fdiv_rn(__fsub_rn(__fsub_rn(z, vz), __fmul_rn(curv, d2)), __fsqrt_rn(d2));
                // the vertex (a, rint(b)) against the steps before this one
                const float zr = r == b0 ? zlo[u] : zhi[u];
                const float mr = hz_vs_metres((float)r, vb, dpc, sb);
                const float d2r = __fadd_rn(__fmul_rn(ma, ma), __fmul_rn(mr, mr));
                const float q = __fdiv_rn(__fadd_rn(__fsub_rn(__fsub_rn(zr, vz), __fmul_rn(curv, d2r)), th), __fsqrt_rn(d2r));
                if(q >= smax)
                {
                    const int i = xmaj ? a : r, j = xmaj ? r : a;
                    word = mask + (size_t)j * p.w32 + (i >> 5);
                    bit = 1u << (i & 31);
                }
                smax = fmaxf(smax, s);
            }
            hz_vs_collect(pend, pbits, word, bit, false, lane);
        }
    }
    hz_vs_collect(pend, pbits, nullptr, 0u, true, lane);
}

cudaError_t hz_launch_viewshed(const HzViewshed& p, int nviews, cudaStream_t stream)
{
    if(nviews <= 0) return cudaSuccess;
    const int warps = 2 * ((p.N + 31) / 32) + 2 * ((p.N - 2 + 31) / 32);
    k_viewshed<<<dim3((unsigned)((warps + HZ_VS_WARPS - 1) / HZ_VS_WARPS), (unsigned)nviews), HZ_VS_WARPS * 32, 0, stream>>>(p);
    return cudaGetLastError();
}

// counts[j][i] += the views' bits of cell (i, j): one thread per cell, the 32 threads of a word share its loads
__global__ void __launch_bounds__(256)
k_viewshed_count(const uint32_t* __restrict__ masks, int nviews, int N, int w32, uint32_t* __restrict__ counts)
{
    const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x), j = (int)blockIdx.y;
    if(i >= N) return;
    const size_t per_view = (size_t)N * w32;
    const uint32_t* m = masks + (size_t)j * w32 + (i >> 5);
    unsigned int c = 0;
    for(int v = 0; v < nviews; v++) c += (__ldg(m + (size_t)v * per_view) >> (i & 31)) & 1u;
    if(c) counts[(size_t)j * N + i] += c;
}

cudaError_t hz_launch_viewshed_count(const uint32_t* masks, int nviews, int N, int w32, uint32_t* counts,
                                     cudaStream_t stream)
{
    if(nviews <= 0) return cudaSuccess;
    k_viewshed_count<<<dim3((unsigned)((N + 255) / 256), (unsigned)N), 256, 0, stream>>>(masks, nviews, N, w32, counts);
    return cudaGetLastError();
}

// ================================================================================================
// k_math_probe (tests only): the projection's two angle functions on arrays of arguments
// ================================================================================================

__global__ void k_math_probe(int n, const float* __restrict__ e, const float* __restrict__ nn, const float* __restrict__ h,
                             const float* __restrict__ d2, float* __restrict__ az, float* __restrict__ el)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if(k >= n) return;
    az[k] = hz_atan2_az(e[k], nn[k]);
    el[k] = hz_atan_el(h[k], d2[k]);
}

cudaError_t hz_launch_math_probe(int n, const float* e, const float* nn, const float* h, const float* d2, float* az, float* el,
                                 cudaStream_t stream)
{
    if(n <= 0) return cudaSuccess;
    k_math_probe<<<(n + 255) / 256, 256, 0, stream>>>(n, e, nn, h, d2, az, el);
    return cudaGetLastError();
}
