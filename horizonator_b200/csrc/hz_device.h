// hz_device.h -- interface between the host side of libhorizonator (hz_api.cpp, hz_dem.cpp) and
// its CUDA kernels (hz_kernels.cu).  Internal; the public C ABI is include/*.h.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

// ---- visibility key --------------------------------------------------------------------------
// One 64-bit word per pixel, resolved with a min() reduction (red.global.min.u64):
//     [63:61] ep   epoch of the render that wrote the key, counting DOWN from 7: a key of an earlier render is larger
//                  than any key of the current one, i.e. it loses every min() and reads as "nothing drawn yet" -- so
//                  the buffer only has to be cleared when the epoch wraps, every eighth render (17 MB of stores per
//                  3600x600 view otherwise)
//     [60:37] q    window depth quantised to 24 bits (the GL_DEPTH_COMPONENT renderbuffer of
//                  horizonator-lib.c:646; smaller = nearer)
//     [36: 8] id   triangle number in the reference's draw order (horizonator-lib.c:496-508):
//                  2*(j*(2R-1)+i) + {0: (j,i),(j+1,i+1),(j+1,i)   1: (j,i),(j,i+1),(j+1,i+1)}   (< 2^29: R <= 7200)
//     [ 7: 0] r8   the fragment's red channel (fragment.glsl:16 after unorm8 conversion)
// min() over keys == GL_LESS with in-order drawing: nearest q wins, equal q -> first drawn wins.
// The result is independent of the order in which threads get to a pixel.
// (Triangle numbers in the queues carry the opt-in level of detail in bits [30:29]; the key only takes the low 29.)
#define HZ_KEY_CLEAR 0xFFFFFFFFFFFFFFFFull   /* epoch 7, q = 0xFFFFFF = cleared depth 1.0 */
#define HZ_Q_MAX     0xFFFFFFu
#define HZ_KEY_Q_SHIFT     37
#define HZ_KEY_EPOCHS      8u

// epoch and depth of a key as one number: what occlusion tests compare (a key of an earlier epoch compares as farther
// than anything)
static __host__ __device__ inline unsigned int hz_key_top(unsigned long long key) { return (unsigned int)(key >> HZ_KEY_Q_SHIFT); }
// the depth a key holds for a render of epoch `ep`: HZ_Q_MAX (cleared) if the key is an earlier render's
static __host__ __device__ inline unsigned int hz_key_q(unsigned long long key, unsigned int ep)
{
    const unsigned int top = hz_key_top(key);
    return (top >> 24) == ep ? (top & HZ_Q_MAX) : HZ_Q_MAX;
}

// ---- tiles as uploaded (raw file bytes) ------------------------------------------------------
struct HzTiles
{
    const uint8_t* tile[4][4];   // [i_lon][j_lat] device pointers to raw .hgt bytes, nullptr = 0
    int origin_cell[2];          // dem.h: origin_dem_cellij
    int ntiles[2];
    int cpd;                     // 1200 / 3600
};

// ---- culling pyramid over the mosaic (built once at init) -------------------------------------
// block (bj,bi) = the 4x4 cells whose south-west vertex is (4bj, 4bi): (min,max) height of its 5x5 vertices
// tile  (tj,ti) = 8x8 blocks = 32x32 cells: (min,max) over its blocks
constexpr int HZ_MAX_OUT     = 8;   // destinations of one resolve (ranks of a wedge-sharded panorama)
constexpr int HZ_BLOCK_CELLS = 4;
constexpr int HZ_TILE_BLOCKS = 8;
constexpr int HZ_TILE_CELLS  = HZ_BLOCK_CELLS * HZ_TILE_BLOCKS;
// The blocks along the far edges of the mesh may reach beyond its last row/column (by up to 3 vertices; with the
// opt-in level of detail by up to a coarse block): the mosaic has this
// many extra (zero) rows, its pitch covers as many extra columns, and the axis tables as many extra entries, so that the
// meshing kernels read those vertices without clamping (their triangles are left out).
constexpr int HZ_MAX_LOD     = 2;                       // opt-in level of detail: blocks of (4 << lod)^2 cells (HzView::lod)
constexpr int HZ_MESH_PAD    = HZ_BLOCK_CELLS << HZ_MAX_LOD;

// ---- counters a render leaves behind (diagnostics; bench.py and the tests read them) -----------
enum HzStat
{
    HZ_STAT_TILES = 0,          // tiles of the bands looked at
    HZ_STAT_TILES_FAR,          //   ... dropped: beyond zfar
    HZ_STAT_TILES_WINDOW,       //   ... dropped: no pixel centre of the target inside their screen box
    HZ_STAT_TILES_OCCLUDED,     //   ... dropped: every pixel of their screen box already holds something nearer
    HZ_STAT_BLOCKS,             // blocks looked at (both passes)
    HZ_STAT_BLOCKS_FAR,
    HZ_STAT_BLOCKS_WINDOW,
    HZ_STAT_BLOCKS_OCCLUDED,
    HZ_STAT_BLOCKS_MESHED,      // blocks whose 32 triangles were projected and tested exactly
    HZ_STAT_TRIANGLES,          // triangles that passed the exact integer tests and went to set-up
    HZ_STAT_BIG_ENTRIES,        // (triangle, sub-box) pairs queued for k_big
    HZ_STAT_COUNT = 16
};

// ---- one render ------------------------------------------------------------------------------
struct alignas(16) HzView      // (16-byte units: the kernels fetch their copy with 128-bit loads, see HZ_KERNEL_PROLOGUE)
{
    // terrain (resident in HBM): N x N int16, row j = north index, column i = east index
    const int16_t* mosaic;       // [N + HZ_MESH_PAD][pitch]
    int   N;                     // 2R
    int   pitch;                 // elements per row (multiple of 64, >= N + HZ_MESH_PAD)
    float* e_tab;                // [N + HZ_MESH_PAD] metres east of the eye for column i   (vertex.glsl:128-130)
    float* n_tab;                // [N + HZ_MESH_PAD] metres north of the eye for row j
    const short2* mm_block;      // [nb][nb] (min,max) per block
    const short2* mm_tile;       // [nt][nt] (min,max) per tile
    int   nb, nt;

    // eye
    float viewer_cell_i, viewer_cell_j, viewer_z;
    float deg_per_cell, cos_viewer_lat;
    float curvature;             // 0 = the reference's flat earth; else apparent height drops by curvature * distance^2
    float seam_period;           // 0 = the reference (triangles across the window's +-pi seam are dropped); else the
                                 // period of x_ndc, az_ndc_per_rad * 2 * pi: such triangles are drawn at both edges

    // azimuth window; scalars the vertex shader derives from az_deg0/az_deg1 (vertex.glsl:139-150),
    // computed once on the host in float exactly as written there
    float az_center;             // az_rad_center
    float az_ndc_per_rad;        // 2/(az_rad1-az_rad0)
    float aspect;                // W/H of the FULL panorama

    float znear, zfar, znear_color, zfar_color;

    // target: the panorama is W x H; this render fills columns [x0, x1) of it
    int W, H;
    int x0, x1;
    unsigned long long* vis;     // [H][x1-x0], GL row order (row 0 = bottom)
    unsigned int epoch;          // of this render's keys (see the visibility key)
    unsigned int clear_keys;     // k_prepare clears this many keys (the whole allocation when the epoch wrapped, else 0)

    // The mesh is walked outwards from the eye.  Tiles within `near_rings` (Chebyshev distance in tiles) of the
    // eye's tile go first and completely (k_near + k_big), then bands of rings [ring_lo, ring_hi), each through
    // k_tiles -> k_blocks -> k_mesh, so that the foreground is in the visibility buffer before what lies behind
    // it is tested against it.
    int eye_ti, eye_tj, near_rings;
    int ring_lo, ring_hi;        // the band this launch works on
    int lod;                     // 0 = the reference's mesh.  Opt-in (horizonator_set_lod): the band is meshed with every
                                 // (1 << lod)-th vertex -- blocks of (4 << lod)^2 cells, still 5x5 vertices and 32 triangles
    uint32_t* tile_queue;        // live tiles of the band (tj << 16 | ti)
    uint32_t* tile_count;
    uint32_t* block_queue;       // live blocks of the band (bj << 16 | bi)
    uint32_t* block_count;
    uint32_t* tri_queue;         // triangles of the stage that passed the exact integer tests
    uint32_t* tri_count;
    uint32_t  tri_capacity;
    int occl_tile_max_pix, occl_block_max_pix;   // largest screen box one thread checks against the visibility buffer
    int grid_percent;            // host only: scale of the device-counted kernels' grids (hz_grid)
    int lod_capable;             // host only: some view of the launch may have lod > 0 (picks k_blocks' instantiation)
    int mid_level;               // host only: the blocks of live tiles are tested in two levels (k_blocks_mid)
    int small_max_pix;           // a lane rasterises bounding boxes up to this many pixels itself; larger ones go to k_big
    int mid_max_pix;             // ... and up to this many where enough lanes of its warp have one (k_raster)

    // triangles too big for one thread: the set-up triangle goes to the record pool (6 x 16 bytes each), and one
    // (record, sub-box) entry per sub-box of its bounding box to a queue -- one queue for the near pass, one for all
    // the bands, one pool for both
    uint2*    big_queue;
    uint32_t* big_count;
    uint32_t  big_capacity;
    uint4*    bigtri;
    uint32_t* bigtri_count;
    uint32_t  bigtri_capacity;
    uint32_t* stats;             // [HZ_STAT_COUNT]

    float cell_diag2;            // (east cell size)^2 + (north cell size)^2 in metres^2, rounded up
    float inv_zrange;            // 1/(zfar-znear), for the conservative depth bound only
    float box_margin;            // pixels added around the screen box of a mesh rectangle (hz_rect_test)

    // k_prepare zeroes these; k_resolve turns the visibility keys into the outputs
    uint32_t* counters;
    int       ncounters;
    const float* tanel;          // [H] tan(elevation) per GL row, host-computed (lib:1007-1012)
    // destinations: normally one, exactly the target ([H][x1-x0], stride x1-x0, offset 0); several (the full
    // panoramas of all ranks, in peer memory) when a wedge-sharded panorama is assembled by the resolve kernel itself.
    // Either pointer of a destination may be null; all destinations have the same ones null.
    int       n_out, out_stride, out_x0;
    uint8_t*  out_image[HZ_MAX_OUT];    // B,G,R top row first
    float*    out_ranges[HZ_MAX_OUT];   // top row first
};

// A render's parameters live in device memory as a small array of HzView variants that differ only in the
// queue/counter/band fields: the kernels take a pointer to their variant, so that the same captured CUDA graph can
// be replayed for every view after one small host->device copy.
enum { HZ_V_NEAR = 0, HZ_V_FAR = 1, HZ_V_BAND0 = 2 };
constexpr int HZ_MAX_BANDS = 14;
constexpr int HZ_V_COUNT   = HZ_V_BAND0 + HZ_MAX_BANDS;

// flags of the GPU-side barrier between the ranks of a wedge-sharded panorama (k_peer_barrier)
struct HzPeerFlags
{
    uint32_t* arrive[HZ_MAX_OUT];    // arrive[r] = rank r's array of HZ_MAX_OUT + 1 words, mapped here
    int n, rank;
};
cudaError_t hz_launch_peer_barrier(const HzPeerFlags& f, unsigned int epoch, cudaStream_t stream);

// All launches are asynchronous on `stream`.  One launch serves `nviews` views at once (gridDim.y = view): `v` is the
// host copy of the variant of view 0 (for grid sizing; every view of a launch has the same image size and band
// structure), `d_v` the device copy of that variant.  View y's copy of the same variant sits HZ_V_COUNT elements
// further per view: d_v + y * HZ_V_COUNT.
cudaError_t hz_launch_mosaic (const HzTiles& t, int16_t* mosaic, int N, int pitch, cudaStream_t stream);
cudaError_t hz_launch_pyramid(const int16_t* mosaic, int N, int pitch, short2* mm_block, int nb,
                              short2* mm_tile, int nt, cudaStream_t stream);
cudaError_t hz_launch_prepare(const HzView& v, const HzView* d_v, int nviews, cudaStream_t stream);  // clear keys, axis tables, counters
cudaError_t hz_launch_near   (const HzView& v, const HzView* d_v, int nviews, cudaStream_t stream);  // foreground tiles -> triangle list
cudaError_t hz_launch_raster (const HzView& v, const HzView* d_v, int nviews, cudaStream_t stream);  // set-up + rasterise a triangle list
cudaError_t hz_launch_band   (const HzView& v, const HzView* d_v, int nviews, bool worst_case, cudaStream_t stream, int* launches);
cudaError_t hz_launch_big    (const HzView& v, const HzView* d_v, int nviews, cudaStream_t stream);  // queued large triangles of one pass
cudaError_t hz_launch_resolve(const HzView& v, const HzView* d_v, int nviews, cudaStream_t stream);
bool        hz_resolve_is_vectorisable(const HzView& v);
cudaError_t hz_launch_horizon(const float* ranges, int n, int W, int H, int* rows, float* range, cudaStream_t stream);
// ---- viewsheds (horizonator_viewshed*: the definition is in include/horizonator-batch.h) ------
constexpr int HZ_VS_MAX_VIEWS = 64;     // views per k_viewshed launch (gridDim.y); their eyes travel in the parameters
struct HzViewshedEye { float vci, vcj, vz, cos_lat; };     // compute_move()'s eye, float as there
struct HzViewshed
{
    const int16_t* mosaic;       // [N + HZ_MESH_PAD][pitch]
    int   N, pitch;
    int   w32;                   // words per mask row, (N + 31) / 32
    float deg_per_cell, curvature, target_height;
    uint32_t* masks;             // view y's mask at masks + y * N * w32, zeroed before the launch
    HzViewshedEye eye[HZ_VS_MAX_VIEWS];
};
cudaError_t hz_launch_viewshed(const HzViewshed& p, int nviews, cudaStream_t stream);
// counts[j * N + i] += the number of the nviews masks (N * w32 words apart) with cell (i, j) set
cudaError_t hz_launch_viewshed_count(const uint32_t* masks, int nviews, int N, int w32, uint32_t* counts,
                                     cudaStream_t stream);

cudaError_t hz_launch_math_probe(int n, const float* e, const float* nn, const float* h, const float* d2, float* az, float* el,
                                 cudaStream_t stream);
