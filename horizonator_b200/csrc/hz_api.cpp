// hz_api.cpp -- the C ABI of include/horizonator.h and include/horizonator-batch.h.
//
// Replaces the host side of /root/reference/horizonator-lib.c: where that file drives an OpenGL context, this
// one owns a block of device state per context (the decoded DEM square, the visibility buffer, output and
// staging buffers, one CUDA stream) and enqueues the kernels of hz_kernels.cu.  The caller-visible struct has
// no room for a pointer, so the state lives in a process-wide table and `ctx->program` holds its handle.
//
// No CPU rendering path exists: without a usable CUDA device horizonator_init() fails.
#include "horizonator.h"
#include "horizonator-batch.h"
#include "util.h"
#include "hz_device.h"

#include <cmath>
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

namespace {

#define CUDA_TRY(expr)                                                              \
    do {                                                                            \
        cudaError_t e__ = (expr);                                                   \
        if(e__ != cudaSuccess)                                                      \
        {                                                                           \
            MSG("CUDA error: %s failed: %s", #expr, cudaGetErrorString(e__));       \
            return false;                                                           \
        }                                                                           \
    } while(0)

constexpr float PI_F            = 3.14159265358979f;       // vertex.glsl:31
// Queue capacities grow with the image (set in alloc_target); whatever does not fit is drawn by a slow in-kernel
// path, so these only have to be generous, not safe.
//   triangles of one stage awaiting set-up:                    max(2^22, pixels/2)
//   (record, sub-box) pairs for the large-triangle kernel:     max(2^21, pixels/4) per pass
//   set-up records of those triangles:                         max(2^18, pixels/16); beyond that k_big repeats the set-up
constexpr int   PROF_EVENTS     = 7;            // 6 stages per render
constexpr int   MAX_BANDS       = HZ_MAX_BANDS;
// [0] big_count near, [1] spare, [2] tri_count near, [3] big-triangle records, [4+4b] tile_count,
// [5+4b] block_count, [6+4b] tri_count, [7+4b] big_count of band b, then the stats
constexpr int   STATS_AT        = 4 + 4 * MAX_BANDS;
constexpr int   N_COUNTERS      = STATS_AT + HZ_STAT_COUNT;

// ---- the render chain's configuration.  Each value won its sweep (profiles/); a new sweep edits a constant and
// compares a second build of the library (build_library(extra_flags, name) + HORIZONATOR_LIBRARY).

constexpr int NEAR_RINGS = 2;                   // rings of tiles around the eye's tile drawn first, without culling tests
// largest bounding box (pixels) a triangle's own thread rasterises always / where enough lanes of its warp have one
// (zoomed-in views only: fill_view); larger ones go to k_big
constexpr int SMALL_MAX_PIX = 16, MID_MAX_PIX = 64;
// most views of a batch rendered by one chain of launches, view sets in flight at once (render_batch_common), and
// executable instances of each captured chain (capture_graph)
constexpr int VIEWS_PER_SET = 64, N_SETS_MAX = 4, GRAPH_INSTANCES = 2;

// Rings (in tiles around the eye's tile) at which the bands end; the last band runs to the edge of the mesh.
struct Bands { int n; int end[MAX_BANDS]; };

// A lone view is latency-bound; the views of a batch want throughput.
// - bands: more bands = more of the mesh culled by what nearer bands drew, but four more kernels each.  A lone view
//   gets two bands.  The views of a batch share their launches -- up to 64 views per chain, so a launch costs next to
//   nothing per view -- and get ten, each reaching about 1.5 times as far as the one before (measured on 256 distinct
//   viewpoints, profiles/r02s_sweep.jsonl: 13.4k panoramas/s with five bands and 16 views per chain, 15.6k with ten
//   and 64; the benchmark viewpoint repeated 30.3k -> 33.0k).  The image is the same either way.
// - occl_tile_max_pix, occl_block_max_pix: largest screen box one thread checks against the visibility buffer.  In a
//   lone view a long walk by one thread holds its kernel up; the views of a batch hide that behind each other and
//   gain from the extra culling.
// - grid_percent: see hz_grid() in hz_kernels.cu.
// - mid_level: blocks of live tiles tested in two levels (k_blocks_mid: fewer tests, one more in a row).
struct ChainConfig { Bands bands; int occl_tile_max_pix, occl_block_max_pix, grid_percent; bool mid_level; };
constexpr ChainConfig LONE  = { { 2, { 48, 1 << 20 } },                                64,  32, 100, false };
constexpr ChainConfig BATCH = { { 10, { 5, 8, 12, 18, 27, 40, 60, 90, 135, 1 << 20 } }, 128, 128, 200, true };
// (with the opt-in level of detail every render has HZ_MAX_LOD more bands: enqueue_views)
static_assert(LONE.bands.n + HZ_MAX_LOD <= HZ_MAX_BANDS && BATCH.bands.n + HZ_MAX_LOD <= HZ_MAX_BANDS, "too many bands");

// what the reference keeps in GL uniforms
struct ViewState
{
    float viewer_cell_i = 0, viewer_cell_j = 0, viewer_z = 0, cos_viewer_lat = 1;
    float az_deg0 = -45.f, az_deg1 = 45.f;
};

constexpr int PARAM_RING = 16;

// which per-row tan(elevation) table a buffer holds (fill_tanel(): a function of the window's width in degrees and of
// the image size only)
struct TanelKey
{
    bool valid = false; float daz = 0; int W = 0, H = 0;
    bool is(float daz_, int W_, int H_) const { return valid && W == W_ && H == H_ && memcmp(&daz, &daz_, sizeof(float)) == 0; }
};

// everything one view in flight writes besides its outputs
struct Scratch
{
    unsigned long long* d_vis = nullptr;
    float *d_e = nullptr, *d_n = nullptr;
    uint32_t *d_tile_queue = nullptr, *d_block_queue = nullptr, *d_tri_queue = nullptr;
    uint2*    d_big_queue = nullptr;   // [2][BIG_CAPACITY]: near pass, bands
    uint4*    d_bigtri = nullptr;      // [BIGTRI_CAPACITY][6]
    uint32_t* d_counters  = nullptr;   // [N_COUNTERS]
    uint8_t*  d_image  = nullptr;      // batch sets only: staging of one view's outputs for the host-pointer batch call
    float*    d_ranges = nullptr;
    // tan(elevation) per row of the window this scratch last rendered (lib:1007-1012; computed on the host like the
    // reference's read-back does, uploaded on the stream of the render that needs it -- so nothing else can be
    // reading the row when it is replaced)
    float*    d_tanel = nullptr;       // [H]
    TanelKey  tanel_key;
    // renders made with this visibility buffer since it was allocated: the epoch of the keys counts down from 7 with it,
    // and the buffer is cleared only when that wraps (hz_device.h, the visibility key)
    unsigned int renders = 0;
    unsigned int last_epoch = 0;       // of the most recent render (horizonator_pick decodes main's keys with it)
};

// Up to `cap` views that are rendered TOGETHER: one chain of kernel launches whose grids have a view dimension
// (gridDim.y), each view with its own scratch.  The context's own view is a set of one; the batch calls use sets of
// up to VIEWS_PER_SET, each with its own stream, so that the tail of one set's kernels overlaps another's.
struct ViewSet
{
    int  cap = 0;
    bool batch = false;                // the chain configuration of batched views (config_of)
    cudaStream_t stream = nullptr;     // batch sets only
    cudaEvent_t  done = nullptr;       // batch sets only
    std::vector<Scratch> sc;           // grows on demand up to cap (ensure_views)

    // parameters of the renders in flight: the kernels read d_views; the host fills a slot of the pinned ring and
    // copies it over (the ring lets several renders be queued without waiting)
    HzView* d_views = nullptr;         // [cap][HZ_V_COUNT]
    HzView* h_views = nullptr;         // pinned [PARAM_RING][cap][HZ_V_COUNT]
    float*  h_tanel = nullptr;         // pinned [PARAM_RING][cap][H] (alloc_target)
    cudaEvent_t ring_ev[PARAM_RING] = {};
    int ring_next = 0;
    cudaEvent_t  busy = nullptr;       // recorded after the last render that used this set
    // the large triangles of the near pass (k_big) are drawn beside the first bands, on a stream of their own
    // (launch_chain): fork after the near pass's k_raster, join before the resolve
    cudaStream_t side = nullptr;
    cudaEvent_t  ev_fork = nullptr, ev_join = nullptr;
    cudaStream_t last_stream = nullptr;
    bool busy_recorded = false;
    // the standard chain, captured on first use per (number of views, shape)
    // (several executable instances each, used in turn: an instance that is still in flight makes the next launch of
    // the SAME instance wait on the host)
    struct Graph { int m; bool big_per_band; std::vector<cudaGraphExec_t> exec; size_t next; int launches; };
    std::vector<Graph> graphs;
    bool graph_failed = false;
};

struct Slot
{
    int device = 0;
    cudaStream_t stream = nullptr;

    // terrain
    int N = 0, pitch = 0, cpd = 0;
    int16_t* d_mosaic = nullptr;
    HzTiles  tiles{};
    short2 *d_mm_block = nullptr, *d_mm_tile = nullptr;   // culling pyramid
    int nb = 0, nt = 0;

    // target
    int W = 0, H = 0;
    uint8_t* d_image  = nullptr;
    float*   d_ranges = nullptr;
    size_t   target_pixels = 0;      // capacity of the buffers above
    uint32_t tri_capacity = 0, big_capacity = 0, bigtri_capacity = 0;

    // page-locked staging for results that go to pageable host memory (copy_to_pageable): made on first use
    char*  h_stage = nullptr;
    size_t h_stage_bytes = 0;
    std::vector<cudaEvent_t> stage_ev;

    // host-side cache of tan(elevation) row tables (tanf() per row is not free; callers re-render the same few windows)
    struct TanelRow { TanelKey key; std::vector<float> row; };
    std::vector<TanelRow> tanel_cache;
    size_t tanel_cache_next = 0;

    // `main` serves the single-view entry points (and keeps the last visibility buffer for horizonator_pick);
    // `sets` are made on demand by the batch entry points.
    ViewSet main;
    std::vector<ViewSet*> sets;
    cudaEvent_t fork_ev = nullptr;

    ViewState view;
    float znear = HORIZONATOR_ZNEAR_DEFAULT, zfar = HORIZONATOR_ZFAR_DEFAULT;
    float znear_color = HORIZONATOR_ZNEAR_DEFAULT, zfar_color = HORIZONATOR_ZFAR_DEFAULT;

    bool have_render = false;        // main's d_vis holds a complete full-width render (for pick)
    unsigned launches_last = 0;

    // optional per-kernel timing: PROF_EVENTS events per recorded render
    bool profiling = false;
    float lod_pixels = 0.f;          // opt-in (horizonator_set_lod); 0 = every band meshed at full density like the reference
    bool  seam_wrap = false;         // opt-in (horizonator_set_seam_wrap); false = seam triangles dropped like the reference
    float curvature = 0.f;           // opt-in (horizonator_set_earth_curvature); 0 = flat earth like the reference
    bool collect_stats = false;      // culling counters (horizonator_render_counters); off: the kernels skip them
    std::vector<cudaEvent_t> prof_events;
    size_t prof_used = 0;

    // viewsheds, allocated by the first viewshed call that needs them: the masks of one chunk of views for calls that
    // want only counts or want the masks in host memory, and the counts of the host-memory call.  A call's stream
    // waits for `vs_done` of the call before it, which may have been queued on another stream and use the same scratch.
    uint32_t* d_vs_masks = nullptr;
    int       vs_mask_views = 0;
    uint32_t* d_vs_counts = nullptr;
    cudaEvent_t vs_done = nullptr;
};

std::mutex          g_table_mutex;
std::vector<Slot*>  g_table;         // handle = index + 1

Slot* slot_of(const horizonator_context_t* ctx)
{
    if(ctx == nullptr || ctx->Ntriangles <= 0 || ctx->program == 0) return nullptr;
    std::lock_guard<std::mutex> lock(g_table_mutex);
    if(ctx->program > g_table.size()) return nullptr;
    return g_table[ctx->program - 1];
}

struct DeviceGuard
{
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev)
    {
        if(cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() { if(prev >= 0) cudaSetDevice(prev); }
};

void drop_graphs(ViewSet& vs)
{
    for(ViewSet::Graph& g : vs.graphs) for(cudaGraphExec_t e : g.exec) cudaGraphExecDestroy(e);
    vs.graphs.clear();
    vs.graph_failed = false;
}

// the part of a scratch whose size depends on the image
void free_scratch_target(Scratch& c)
{
    cudaFree(c.d_vis); cudaFree(c.d_image); cudaFree(c.d_ranges);
    cudaFree(c.d_tri_queue); cudaFree(c.d_big_queue); cudaFree(c.d_bigtri); cudaFree(c.d_tanel);
    c.d_vis = nullptr; c.d_image = nullptr; c.d_ranges = nullptr;
    c.d_tri_queue = nullptr; c.d_big_queue = nullptr; c.d_bigtri = nullptr; c.d_tanel = nullptr;
    c.tanel_key = TanelKey{};
    c.renders = 0;
}

bool alloc_scratch_target(const Slot& s, Scratch& c, bool staging)
{
    const size_t px = s.target_pixels;
    CUDA_TRY(cudaMalloc(&c.d_vis, px * sizeof(unsigned long long)));
    CUDA_TRY(cudaMalloc(&c.d_tri_queue, (size_t)s.tri_capacity * sizeof(uint32_t)));
    CUDA_TRY(cudaMalloc(&c.d_big_queue, 2 * (size_t)s.big_capacity * sizeof(uint2)));
    CUDA_TRY(cudaMalloc(&c.d_bigtri, (size_t)s.bigtri_capacity * 6 * sizeof(uint4)));
    CUDA_TRY(cudaMalloc(&c.d_tanel, (size_t)s.H * sizeof(float)));
    if(staging)
    {
        CUDA_TRY(cudaMalloc(&c.d_image, px * 3));
        CUDA_TRY(cudaMalloc(&c.d_ranges, px * sizeof(float)));
    }
    return true;
}

void free_set_target(ViewSet& vs)
{
    drop_graphs(vs);
    for(Scratch& c : vs.sc) free_scratch_target(c);
    cudaFreeHost(vs.h_tanel); vs.h_tanel = nullptr;
}

bool alloc_set_target(const Slot& s, ViewSet& vs)
{
    CUDA_TRY(cudaMallocHost(&vs.h_tanel, (size_t)PARAM_RING * vs.cap * s.H * sizeof(float)));
    for(Scratch& c : vs.sc) if(!alloc_scratch_target(s, c, vs.batch)) return false;
    return true;
}

void free_target(Slot& s)
{
    free_set_target(s.main);
    for(ViewSet* g : s.sets) free_set_target(*g);
    cudaFree(s.d_image);  s.d_image = nullptr;
    cudaFree(s.d_ranges); s.d_ranges = nullptr;
    cudaFreeHost(s.h_stage); s.h_stage = nullptr; s.h_stage_bytes = 0;
    for(cudaEvent_t e : s.stage_ev) cudaEventDestroy(e);
    s.stage_ev.clear();
    s.target_pixels = 0;
    s.tanel_cache.clear();
}

// A failure part way leaves the context without a target (W = H = 0): later renders return false instead of
// running kernels on buffers that are not there.
bool alloc_target(Slot& s, int W, int H)
{
    free_target(s);
    s.W = 0; s.H = 0; s.have_render = false;
    const size_t px = (size_t)W * (size_t)H;
    auto cap = [px](size_t floor_, size_t div) {
        const size_t c = px / div > floor_ ? px / div : floor_;
        return (uint32_t)(c > 0x7FFFFFFFu ? 0x7FFFFFFFu : c);
    };
    s.tri_capacity = cap((size_t)1 << 22, 2); s.big_capacity = cap((size_t)1 << 21, 4); s.bigtri_capacity = cap((size_t)1 << 18, 16);
    // tests shrink the queues to exercise the overflow paths
    if(const char* env = getenv("HORIZONATOR_TRI_CAPACITY"))    s.tri_capacity    = (uint32_t)(atoi(env) > 1 ? atoi(env) : 1);
    if(const char* env = getenv("HORIZONATOR_BIG_CAPACITY"))    s.big_capacity    = (uint32_t)(atoi(env) > 1 ? atoi(env) : 1);
    if(const char* env = getenv("HORIZONATOR_BIGTRI_CAPACITY")) s.bigtri_capacity = (uint32_t)(atoi(env) > 1 ? atoi(env) : 1);
    s.target_pixels = px; s.W = W; s.H = H;       // alloc_*_target() size their buffers from these
    bool ok = alloc_set_target(s, s.main);
    for(ViewSet* g : s.sets) ok = ok && alloc_set_target(s, *g);
    ok = ok && cudaMalloc(&s.d_image, px * 3) == cudaSuccess && cudaMalloc(&s.d_ranges, px * sizeof(float)) == cudaSuccess;
    if(!ok)
    {
        MSG("Could not allocate the %d x %d render target", W, H);
        cudaGetLastError();
        free_target(s);
        s.W = 0; s.H = 0;
        return false;
    }
    return true;
}

void free_scratch(Scratch& c)
{
    free_scratch_target(c);
    cudaFree(c.d_e); cudaFree(c.d_n);
    cudaFree(c.d_tile_queue); cudaFree(c.d_block_queue);
    cudaFree(c.d_counters);
    c = Scratch{};
}

// everything but the image-sized part (alloc_scratch_target)
bool alloc_scratch(const Slot& s, Scratch& c)
{
    CUDA_TRY(cudaMalloc(&c.d_e, (size_t)(s.N + HZ_MESH_PAD) * sizeof(float)));
    CUDA_TRY(cudaMalloc(&c.d_n, (size_t)(s.N + HZ_MESH_PAD) * sizeof(float)));
    CUDA_TRY(cudaMalloc(&c.d_tile_queue, (size_t)s.nt * s.nt * sizeof(uint32_t)));
    CUDA_TRY(cudaMalloc(&c.d_block_queue, (size_t)s.nb * s.nb * sizeof(uint32_t)));
    CUDA_TRY(cudaMalloc(&c.d_counters, N_COUNTERS * sizeof(uint32_t)));
    return true;
}

void free_set(ViewSet& vs)
{
    free_set_target(vs);
    for(Scratch& c : vs.sc) free_scratch(c);
    vs.sc.clear();
    cudaFree(vs.d_views); cudaFreeHost(vs.h_views);
    for(cudaEvent_t e : vs.ring_ev) if(e) cudaEventDestroy(e);
    if(vs.busy) cudaEventDestroy(vs.busy);
    if(vs.ev_fork) cudaEventDestroy(vs.ev_fork);
    if(vs.ev_join) cudaEventDestroy(vs.ev_join);
    if(vs.side) cudaStreamDestroy(vs.side);
    if(vs.done) cudaEventDestroy(vs.done);
    if(vs.stream) cudaStreamDestroy(vs.stream);
    vs = ViewSet{};
}

// the set's own resources; its scratches come with ensure_views()
bool alloc_set(ViewSet& vs, int cap, bool batch)
{
    vs.cap = cap; vs.batch = batch;
    CUDA_TRY(cudaMalloc(&vs.d_views, (size_t)cap * HZ_V_COUNT * sizeof(HzView)));
    CUDA_TRY(cudaMallocHost(&vs.h_views, (size_t)PARAM_RING * cap * HZ_V_COUNT * sizeof(HzView)));
    for(cudaEvent_t& e : vs.ring_ev) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&vs.busy, cudaEventDisableTiming));
    if(batch)
    {
        CUDA_TRY(cudaStreamCreateWithFlags(&vs.stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&vs.done, cudaEventDisableTiming));
    }
    return true;
}

// bytes of device memory one scratch takes (what ensure_views() budgets with)
size_t scratch_bytes(const Slot& s)
{
    const size_t px = s.target_pixels;
    return px * (sizeof(unsigned long long) + 3 + sizeof(float)) +
           ((size_t)s.tri_capacity + (size_t)s.nt * s.nt + (size_t)s.nb * s.nb + 2 * (size_t)s.N) * sizeof(uint32_t) +
           2 * (size_t)s.big_capacity * sizeof(uint2) + (size_t)s.bigtri_capacity * 6 * sizeof(uint4);
}

// Makes sure the set has scratch for up to n views (n <= cap) and returns how many it has to use.  Batch sets only
// grow while the new scratch fits into half of the device memory that is free right now (a 36000 x 4000 panorama
// needs ~3 GB per view in flight).
int ensure_views(Slot& s, ViewSet& vs, int n)
{
    if(n > vs.cap) n = vs.cap;
    while((int)vs.sc.size() < n)
    {
        if(vs.batch)
        {
            size_t free_b = 0, total_b = 0;
            if(cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || scratch_bytes(s) > free_b / 2) break;
        }
        Scratch c;
        if(!alloc_scratch(s, c) || (s.target_pixels > 0 && !alloc_scratch_target(s, c, vs.batch)))
        {
            MSG("Could not allocate the scratch of view %d of a set", (int)vs.sc.size());
            cudaGetLastError();
            free_scratch(c);
            break;
        }
        vs.sc.push_back(c);
    }
    return (int)vs.sc.size() < n ? (int)vs.sc.size() : n;
}

// the batch sets: up to N_SETS_MAX, created on demand
ViewSet* batch_set(Slot& s, int k)
{
    if(s.fork_ev == nullptr && cudaEventCreateWithFlags(&s.fork_ev, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    while((int)s.sets.size() <= k)
    {
        ViewSet* g = new ViewSet;
        bool ok = alloc_set(*g, VIEWS_PER_SET, true);
        if(ok && s.target_pixels > 0)
            ok = cudaMallocHost(&g->h_tanel, (size_t)PARAM_RING * g->cap * s.H * sizeof(float)) == cudaSuccess;
        if(!ok)
        {
            MSG("Could not allocate view set %d", (int)s.sets.size());
            cudaGetLastError();
            free_set(*g);
            delete g;
            return nullptr;
        }
        s.sets.push_back(g);
    }
    return s.sets[k];
}

void destroy_slot(Slot* s)
{
    if(s == nullptr) return;
    DeviceGuard g(s->device);
    if(s->stream) cudaStreamSynchronize(s->stream);
    for(ViewSet* v : s->sets) if(v->stream) cudaStreamSynchronize(v->stream);
    free_target(*s);
    free_set(s->main);
    for(ViewSet* v : s->sets) { free_set(*v); delete v; }
    if(s->fork_ev) cudaEventDestroy(s->fork_ev);
    cudaFree(s->d_mosaic);
    for(int i = 0; i < 4; i++) for(int j = 0; j < 4; j++) cudaFree((void*)s->tiles.tile[i][j]);
    for(cudaEvent_t e : s->prof_events) cudaEventDestroy(e);
    cudaFree(s->d_mm_block); cudaFree(s->d_mm_tile);
    if(s->vs_done) { cudaEventSynchronize(s->vs_done); cudaEventDestroy(s->vs_done); }
    cudaFree(s->d_vs_masks); cudaFree(s->d_vs_counts);
    if(s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

// vertex.glsl:34-38 on the host, in float (round() = round-half-even, oracle rule F9)
float unwrap_near_rad(float x, float near)
{
    const float d = (x - near) / (2.f * PI_F);
    return (d - rintf(d)) * 2.f * PI_F + near;
}

// lib:1007-1012: tan(elevation) of each GL row as the reference's read-back computes it -- rows of the
// lower half directly, rows of the upper half as the negated value of their mirror row.
void fill_tanel(float* out, int W, int H, float az_deg0, float az_deg1)
{
    const float aspect = (float)W / (float)H;
    for(int y = 0; y < H; y++)
    {
        const int   ysrc   = (y < H / 2 || ((H & 1) && y == H / 2)) ? y : H - 1 - y;
        const float el_ndc = ((float)ysrc + 0.5f) / (float)H * 2.f - 1.f;
        const float el     = el_ndc * (az_deg1 - az_deg0) / 2.f / aspect * M_PI / 180.0f;
        const float t      = tanf(el);
        out[y] = (ysrc != y) ? -t : t;
    }
}

// the row table of a window from the host cache, computing it if it is not there
const float* tanel_row(Slot& s, float az_deg0, float az_deg1)
{
    const float daz = az_deg1 - az_deg0;
    for(const Slot::TanelRow& r : s.tanel_cache) if(r.key.is(daz, s.W, s.H)) return r.row.data();
    constexpr size_t CACHE = 64;
    if(s.tanel_cache.size() < CACHE) { s.tanel_cache.emplace_back(); s.tanel_cache_next = s.tanel_cache.size() - 1; }
    else s.tanel_cache_next = (s.tanel_cache_next + 1) % CACHE;
    Slot::TanelRow& r = s.tanel_cache[s.tanel_cache_next];
    r.row.resize((size_t)s.H);
    fill_tanel(r.row.data(), s.W, s.H, az_deg0, az_deg1);
    r.key.valid = true; r.key.daz = daz; r.key.W = s.W; r.key.H = s.H;
    return r.row.data();
}

const ChainConfig& config_of(const ViewSet& set)
{
    return set.batch ? BATCH : LONE;
}

// bands of a render chain: the configured ones, plus two more where the opt-in level of detail changes (fill: enqueue_views)
int n_bands_of(const Slot& s, const ViewSet& set)
{
    return config_of(set).bands.n + (s.lod_pixels > 0.f ? HZ_MAX_LOD : 0);
}

// Zoomed-in views (small angle per pixel) show triangles many pixels large even far from the eye: each band then draws
// its large triangles before the next band is tested against the visibility buffer.  In wide views the far bands have
// hardly any, and one k_big after the last band saves a launch per band.
bool big_after_every_band(const Slot& s, const ViewState& vs)
{
    return fabsf(vs.az_deg1 - vs.az_deg0) < 0.05f * (float)s.W;
}

// the kernels of one render of m views, in order, reading their parameters from set.d_views; hv = the host copy of those
bool launch_chain(Slot& s, ViewSet& set, const HzView* hv, int m, bool big_per_band, bool worst_case, bool resolve,
                  cudaStream_t st, cudaEvent_t* ev, int* launches)
{
    const HzView* dv = set.d_views;
    int n = 0;
    if(ev) CUDA_TRY(cudaEventRecord(ev[0], st));
    CUDA_TRY(hz_launch_prepare(hv[HZ_V_NEAR], dv + HZ_V_NEAR, m, st)); n++;
    if(ev) CUDA_TRY(cudaEventRecord(ev[1], st));
    CUDA_TRY(hz_launch_near(hv[HZ_V_NEAR], dv + HZ_V_NEAR, m, st)); n++;
    CUDA_TRY(hz_launch_raster(hv[HZ_V_NEAR], dv + HZ_V_NEAR, m, st)); n++;
    if(ev) CUDA_TRY(cudaEventRecord(ev[2], st));
    // The near pass's large triangles: in line, or (fork) beside the bands on the set's side stream.  The bands' culling
    // then sees less of the foreground in the visibility buffer -- it only ever removes work, the image is the same --
    // and the chain is a kernel shorter.  Measured on one box against the chain in line: lone C2 view 111 -> 108 us,
    // 10-degree zoom 0.38 -> 0.35 ms, 5-degree 0.28 -> 0.25 ms, eye 12 km +1 %, batches +0.5 %.  A profiled chain
    // (ev) runs it in line, so that the events time each kernel.
    const bool fork = ev == nullptr;
    if(fork && set.side == nullptr)
    {
        CUDA_TRY(cudaEventCreateWithFlags(&set.ev_fork, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&set.ev_join, cudaEventDisableTiming));
        CUDA_TRY(cudaStreamCreateWithFlags(&set.side, cudaStreamNonBlocking));
    }
    if(fork)
    {
        CUDA_TRY(cudaEventRecord(set.ev_fork, st));
        CUDA_TRY(cudaStreamWaitEvent(set.side, set.ev_fork, 0));
        CUDA_TRY(hz_launch_big(hv[HZ_V_NEAR], dv + HZ_V_NEAR, m, set.side)); n++;
        CUDA_TRY(cudaEventRecord(set.ev_join, set.side));
    }
    else { CUDA_TRY(hz_launch_big(hv[HZ_V_NEAR], dv + HZ_V_NEAR, m, st)); n++; }
    if(ev) CUDA_TRY(cudaEventRecord(ev[3], st));
    const int n_bands = n_bands_of(s, set);
    for(int b = 0; b < n_bands; b++)
    {
        const bool last = (b + 1 == n_bands);
        int k = 0;
        CUDA_TRY(hz_launch_band(hv[HZ_V_BAND0 + b], dv + HZ_V_BAND0 + b, m, worst_case, st, &k));
        n += k;
        if(last && ev) CUDA_TRY(cudaEventRecord(ev[4], st));
        // all bands share one queue and counter unless every band has its own k_big (see fill_views)
        if(last || (big_per_band && k > 0)) { CUDA_TRY(hz_launch_big(hv[HZ_V_BAND0 + b], dv + HZ_V_BAND0 + b, m, st)); n++; }
    }
    if(ev) CUDA_TRY(cudaEventRecord(ev[5], st));
    if(fork) CUDA_TRY(cudaStreamWaitEvent(st, set.ev_join, 0));
    if(resolve) { CUDA_TRY(hz_launch_resolve(hv[HZ_V_NEAR], dv + HZ_V_NEAR, m, st)); n++; }
    if(ev) CUDA_TRY(cudaEventRecord(ev[6], st));
    *launches = n;
    return true;
}

// Captures the standard chain (full width, vectorised resolve, grids sized for any eye position) for m views of the
// set; every later standard render of m views is one cudaGraphLaunch after the parameter copy.  A dozen separate
// launches cost more host time than the GPU needs for the render.
ViewSet::Graph* capture_graph(Slot& s, ViewSet& set, const HzView* hv, int m, bool big_per_band)
{
    cudaStream_t cs = nullptr;
    if(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    cudaGraph_t g = nullptr;
    std::vector<cudaGraphExec_t> exec;
    bool ok = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    int launches = 0;
    if(ok)
    {
        ok = launch_chain(s, set, hv, m, big_per_band, true, true, cs, nullptr, &launches);
        if(cudaStreamEndCapture(cs, &g) != cudaSuccess) ok = false;
    }
    for(int k = 0; ok && k < GRAPH_INSTANCES; k++)
    {
        cudaGraphExec_t e = nullptr;
        if(cudaGraphInstantiate(&e, g, 0) != cudaSuccess) ok = false; else exec.push_back(e);
    }
    if(!ok) for(cudaGraphExec_t e : exec) cudaGraphExecDestroy(e);
    if(g) cudaGraphDestroy(g);
    cudaStreamDestroy(cs);
    if(!ok)
    {
        cudaGetLastError();
        MSG("CUDA graph capture of the render chain failed; launching the kernels one by one instead");
        return nullptr;
    }
    set.graphs.push_back(ViewSet::Graph{ m, big_per_band, exec, 0, launches });
    return &set.graphs.back();
}

// where a render's outputs go (see HzView::n_out): one destination shaped like the target, or the full panoramas
// of several ranks
struct OutSpec
{
    int n = 1;
    uint8_t* image[HZ_MAX_OUT] = {};
    float*   ranges[HZ_MAX_OUT] = {};
    int stride = 0;              // pixels per destination row; 0 = the target's own width (x1-x0)
    int x_off = 0;               // column of the destination where the target's first column goes
};

OutSpec single_out(uint8_t* d_image, float* d_ranges)
{
    OutSpec o;
    o.image[0] = d_image; o.ranges[0] = d_ranges;
    return o;
}

// the parameters of one view: everything but the queue/counter/band fields that differ between the variants
void fill_view(const Slot& s, const ViewSet& set, const Scratch& sc, const ViewState& vs, int x0, int x1, const OutSpec& out,
               HzView& v)
{
    v = HzView{};
    v.mosaic = s.d_mosaic; v.N = s.N; v.pitch = s.pitch;
    v.e_tab = sc.d_e; v.n_tab = sc.d_n;
    v.mm_block = s.d_mm_block; v.nb = s.nb;
    v.mm_tile  = s.d_mm_tile;  v.nt = s.nt;
    v.viewer_cell_i = vs.viewer_cell_i; v.viewer_cell_j = vs.viewer_cell_j; v.viewer_z = vs.viewer_z;
    v.deg_per_cell = 1.0f / (float)s.cpd;                                // lib:577
    v.cos_viewer_lat = vs.cos_viewer_lat;
    v.curvature = s.curvature;

    // vertex.glsl:139-150, float
    const float az_rad0 = vs.az_deg0 * 0.017453292519943295f;            // radians()
    float       az_rad1 = vs.az_deg1 * 0.017453292519943295f;
    az_rad1 = unwrap_near_rad(az_rad1 - az_rad0, PI_F) + az_rad0;
    v.az_center      = (az_rad0 + az_rad1) / 2.f;
    v.az_ndc_per_rad = 2.0f / (az_rad1 - az_rad0);
    v.aspect         = (float)s.W / (float)s.H;                          // lib:658-659
    v.seam_period    = s.seam_wrap ? v.az_ndc_per_rad * 2.f * PI_F : 0.0f;

    v.znear = s.znear; v.zfar = s.zfar; v.znear_color = s.znear_color; v.zfar_color = s.zfar_color;
    v.W = s.W; v.H = s.H; v.x0 = x0; v.x1 = x1;
    v.vis = sc.d_vis;
    v.stats      = s.collect_stats ? sc.d_counters + STATS_AT : nullptr;
    v.tile_queue = sc.d_tile_queue; v.block_queue = sc.d_block_queue;
    v.tri_queue = sc.d_tri_queue; v.tri_capacity = s.tri_capacity;
    v.bigtri = sc.d_bigtri; v.bigtri_count = sc.d_counters + 3; v.bigtri_capacity = s.bigtri_capacity;
    const ChainConfig& cfg = config_of(set);
    v.occl_tile_max_pix  = cfg.occl_tile_max_pix;
    v.occl_block_max_pix = cfg.occl_block_max_pix;
    // (middle-sized triangles are drawn by their own threads only in zoomed-in views, where whole warps have them; in a
    // wide view they sit right around the eye, and walking them in k_raster holds that kernel up for nothing)
    // (... and in such views the threads walk boxes twice as large themselves: measured 5 % faster)
    const bool zoomed = big_after_every_band(s, vs);
    v.small_max_pix = zoomed ? 2 * SMALL_MAX_PIX : SMALL_MAX_PIX; v.mid_max_pix = zoomed ? MID_MAX_PIX : 0;
    v.grid_percent = cfg.grid_percent;
    v.lod_capable = s.lod_pixels > 0.f;
    v.mid_level = cfg.mid_level;
    v.big_capacity = s.big_capacity;

    // the eye's tile, and how many rings of tiles around it form the foreground pass
    {
        const int ti = (int)floorf(vs.viewer_cell_i / (float)HZ_TILE_CELLS), tj = (int)floorf(vs.viewer_cell_j / (float)HZ_TILE_CELLS);
        v.eye_ti = ti < 0 ? 0 : (ti >= s.nt ? s.nt - 1 : ti);
        v.eye_tj = tj < 0 ? 0 : (tj >= s.nt ? s.nt - 1 : tj);
        v.near_rings = NEAR_RINGS;
    }

    // for the depth bound of hz_rect_test: the diagonal of one cell on the ground
    {
        const double cn = (double)v.deg_per_cell * 6371000.0 * M_PI / 180.0, ce = cn * fabs((double)vs.cos_viewer_lat);
        v.cell_diag2 = (float)((ce * ce + cn * cn) * 1.01);
        // 1/64 pixel for snapping (1/512) and the few-ulp wobble of the angle functions, plus 8 float ulps of the
        // largest window coordinate (an ulp of x at column 36000 is already 1/256 pixel)
        v.box_margin = 0.015625f + 8.0f * 6e-8f * (float)(s.W > s.H ? s.W : s.H);
        v.inv_zrange = (s.zfar > s.znear) ? 1.0f / (s.zfar - s.znear) : 0.0f;   // 0: no far/occlusion culling
    }

    v.counters = sc.d_counters; v.ncounters = N_COUNTERS;
    v.tanel = sc.d_tanel;
    v.n_out = out.n; v.out_stride = out.stride > 0 ? out.stride : x1 - x0; v.out_x0 = out.x_off;
    for(int d = 0; d < out.n; d++) { v.out_image[d] = out.image[d]; v.out_ranges[d] = out.ranges[d]; }
}

// Enqueues one render of columns [x0,x1) of m views (m <= what ensure_views() gave) on stream st: view k uses scratch
// set.sc[k] and writes to outs[k] (device memory).  All views of one call must have the same kinds of output.
bool enqueue_views(Slot& s, ViewSet& set, int m, const ViewState* vs, int x0, int x1, const OutSpec* outs, cudaStream_t st)
{
    if(s.W <= 0 || s.H <= 0 || m < 1 || m > (int)set.sc.size()) return false;
    const bool want_image = outs[0].image[0] != nullptr, want_ranges = outs[0].ranges[0] != nullptr;
    // a set serves one render at a time: if its previous render went to another stream, wait for that one
    if(set.busy_recorded && set.last_stream != st) CUDA_TRY(cudaStreamWaitEvent(st, set.busy, 0));

    // ---- the parameter block: per view, variants for the near pass, the far queue and each band, into a slot of the
    // pinned ring, then one small copy to the device
    const int slot = set.ring_next;
    set.ring_next = (set.ring_next + 1) % PARAM_RING;
    CUDA_TRY(cudaEventSynchronize(set.ring_ev[slot]));            // the copies that last used this slot are done
    HzView* hv = set.h_views + (size_t)slot * set.cap * HZ_V_COUNT;
    const Bands& bands = config_of(set).bands;
    bool big_per_band = false, vectorisable = true;
    for(int k = 0; k < m; k++) big_per_band = big_per_band || big_after_every_band(s, vs[k]);
    for(int k = 0; k < m; k++)
    {
        Scratch& sc = set.sc[k];
        HzView* hk = hv + (size_t)k * HZ_V_COUNT;
        fill_view(s, set, sc, vs[k], x0, x1, outs[k], hk[0]);
        // the epoch of this render's keys; a fresh or wrapped buffer is cleared first, all of it
        hk[0].epoch = HZ_KEY_EPOCHS - 1u - sc.renders % HZ_KEY_EPOCHS;
        hk[0].clear_keys = (sc.renders % HZ_KEY_EPOCHS == 0) ? (unsigned int)s.target_pixels : 0u;
        sc.last_epoch = hk[0].epoch;
        sc.renders++;
        vectorisable = vectorisable && hz_resolve_is_vectorisable(hk[0]);
        for(int j = 1; j < HZ_V_COUNT; j++) hk[j] = hk[0];
        hk[HZ_V_NEAR].tri_count = sc.d_counters + 2;
        hk[HZ_V_NEAR].big_queue = sc.d_big_queue;                 hk[HZ_V_NEAR].big_count = sc.d_counters + 0;
        for(int j = HZ_V_FAR; j < HZ_V_COUNT; j++)
        {
            hk[j].big_queue = sc.d_big_queue + s.big_capacity;      hk[j].big_count = sc.d_counters + 1;
        }
        // The bands: the configured ring limits -- plus, with the opt-in level of detail, the two rings from which on a
        // cell of 2x2 / 4x4 DEM cells, seen from that ring's nearest edge, is at most lod_pixels pixels across: the level
        // is then the same throughout a band, and the image does not depend on how the bands were configured.
        int ends[HZ_MAX_BANDS], n_ends = 0;
        for(int b = 0; b < bands.n; b++) ends[n_ends++] = bands.end[b];
        int lod_from[HZ_MAX_LOD + 1] = { 0, 1 << 30, 1 << 30 };
        if(s.lod_pixels > 0.f)
        {
            // cell / distance * pixels per radian, distance = (ring - 1) tiles of HZ_TILE_CELLS cells
            const double k_px = fabs((double)hk[0].az_ndc_per_rad) * 0.5 * (double)s.W / (double)HZ_TILE_CELLS;
            for(int l = 1; l <= HZ_MAX_LOD; l++)
            {
                const double r = ceil(k_px * (double)(1 << l) / (double)s.lod_pixels) + 1.0;
                lod_from[l] = r < 2.0 ? 2 : (r > 1e9 ? 1 << 30 : (int)r);
                int at = n_ends;
                while(at > 0 && ends[at - 1] > lod_from[l]) { ends[at] = ends[at - 1]; at--; }
                ends[at] = lod_from[l];
                n_ends++;
            }
        }
        int lo = NEAR_RINGS + 1;
        for(int b = 0; b < n_ends; b++)
        {
            HzView& vb = hk[HZ_V_BAND0 + b];
            vb.ring_lo = lo; vb.ring_hi = ends[b] > lo ? ends[b] : lo;
            vb.tile_count = sc.d_counters + 4 + 4 * b; vb.block_count = sc.d_counters + 5 + 4 * b;
            vb.tri_count  = sc.d_counters + 6 + 4 * b;
            // one k_big per band: each band counts its own entries from 0 (the queue memory is reused, the bands run
            // one after the other); one k_big at the end: all bands append to the same count
            vb.big_count  = sc.d_counters + 7 + (big_per_band ? 4 * b : 0);
            int lod = 0;
            while(lod < HZ_MAX_LOD && vb.ring_lo >= lod_from[lod + 1]) lod++;
            vb.lod = lod;
            vb.cell_diag2 = hk[0].cell_diag2 * (float)((1 << lod) * (1 << lod));
            lo = vb.ring_hi;
        }
        // the row table of this view's window, unless the scratch still holds it from its previous render
        if(want_ranges && !sc.tanel_key.is(vs[k].az_deg1 - vs[k].az_deg0, s.W, s.H))
        {
            float* h_row = set.h_tanel + ((size_t)slot * set.cap + k) * s.H;
            memcpy(h_row, tanel_row(s, vs[k].az_deg0, vs[k].az_deg1), (size_t)s.H * sizeof(float));
            CUDA_TRY(cudaMemcpyAsync(sc.d_tanel, h_row, (size_t)s.H * sizeof(float), cudaMemcpyHostToDevice, st));
            sc.tanel_key.valid = true; sc.tanel_key.daz = vs[k].az_deg1 - vs[k].az_deg0; sc.tanel_key.W = s.W; sc.tanel_key.H = s.H;
        }
    }
    CUDA_TRY(cudaMemcpyAsync(set.d_views, hv, (size_t)m * HZ_V_COUNT * sizeof(HzView), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaEventRecord(set.ring_ev[slot], st));

    // ---- the kernels: a replay of the captured graph where the chain has its standard shape, one by one otherwise
    const bool is_main = (&set == &s.main);
    const bool standard = !s.profiling && x0 == 0 && x1 == s.W && (want_image || want_ranges) &&
                          outs[0].n == 1 && hv[0].out_stride == s.W && outs[0].x_off == 0 && vectorisable;
    if(standard && !set.graph_failed)
    {
        ViewSet::Graph* g = nullptr;
        for(ViewSet::Graph& c : set.graphs) if(c.m == m && c.big_per_band == big_per_band) g = &c;
        if(g == nullptr && (g = capture_graph(s, set, hv, m, big_per_band)) == nullptr) set.graph_failed = true;
        if(g != nullptr)
        {
            CUDA_TRY(cudaGraphLaunch(g->exec[g->next], st));
            g->next = (g->next + 1) % g->exec.size();
            CUDA_TRY(cudaEventRecord(set.busy, st)); set.last_stream = st; set.busy_recorded = true;
            s.launches_last = g->launches;
            if(is_main) s.have_render = true;
            return true;
        }
    }

    cudaEvent_t* ev = nullptr;
    if(s.profiling)
    {
        while(s.prof_events.size() < s.prof_used + PROF_EVENTS)
        {
            cudaEvent_t e;
            CUDA_TRY(cudaEventCreate(&e));
            s.prof_events.push_back(e);
        }
        ev = &s.prof_events[s.prof_used];
        s.prof_used += PROF_EVENTS;
    }
    int launches = 0;
    // grids sized for this view's eye tile only when there is just one view
    if(!launch_chain(s, set, hv, m, big_per_band, m > 1, want_image || want_ranges, st, ev, &launches)) return false;
    CUDA_TRY(cudaEventRecord(set.busy, st)); set.last_stream = st; set.busy_recorded = true;
    s.launches_last = launches;
    if(is_main) s.have_render = (x0 == 0 && x1 == s.W);
    return true;
}

// one view on the context's own scratch
bool enqueue_render(Slot& s, const ViewState& vs, int x0, int x1, const OutSpec& out, cudaStream_t st)
{
    return enqueue_views(s, s.main, 1, &vs, x0, x1, &out, st);
}

// lib:765-789, float as written there.  The four samples come from the host mmaps (dem.h).
bool compute_move(const horizonator_context_t* ctx, float* viewer_z, float lat, float lon, ViewState& vs)
{
    const horizonator_dem_context_t* d = &ctx->dems;
    const float vci = (lon - (float)d->origin_dem_lon_lat[0]) * (float)d->cells_per_deg - (float)d->origin_dem_cellij[0];
    const float vcj = (lat - (float)d->origin_dem_lon_lat[1]) * (float)d->cells_per_deg - (float)d->origin_dem_cellij[1];
    const int i0 = (int)floorf(vci), j0 = (int)floorf(vcj);
    float z;
    if(viewer_z == nullptr || *viewer_z < 0)
    {
        // a little above the ground so that the bumps right next to the eye don't fill the view
        z = (float)((double)fmaxf(fmaxf((float)horizonator_dem_sample(d, i0,     j0),
                                        (float)horizonator_dem_sample(d, i0 + 1, j0)),
                                  fmaxf((float)horizonator_dem_sample(d, i0,     j0 + 1),
                                        (float)horizonator_dem_sample(d, i0 + 1, j0 + 1))) + 1.0);
        if(viewer_z != nullptr) *viewer_z = z;
    }
    else
        z = *viewer_z;
    vs.viewer_cell_i  = vci;
    vs.viewer_cell_j  = vcj;
    vs.viewer_z       = z;
    vs.cos_viewer_lat = cosf((float)((double)lat * M_PI / (double)180.0f));   // lib:799
    return true;
}

// ---- results into pageable host memory ------------------------------------------------------------------------
//
// What an unmodified caller of the reference passes to horizonator_render_offscreen() is ordinary pageable memory
// (horizonator-pywrap.c:234-250 allocates fresh numpy arrays for every render).  A device->host copy into such memory
// goes through a page-locked staging buffer one way or another; the driver's own staging moves a 15 MB result at about
// a third of the PCIe rate, single-threaded.  Here the result is copied in chunks into the context's page-locked
// staging buffer, an event after each chunk, and a few host threads (this one and a small process-wide pool) copy each
// chunk on to the caller's memory as soon as its event has fired: the DMA and the memcpys overlap, and the memcpys
// (and the page faults of a freshly allocated destination) run in parallel.

class HostCopyPool
{
public:
    struct Part { char* dst; const char* src; size_t bytes; cudaEvent_t ready; };

    // copies every part (after its event) with the pool's threads and the calling one; returns when all are done:
    // false if waiting for some part's event failed (that part was not copied)
    bool run(int device, const std::vector<Part>& parts)
    {
        std::unique_lock<std::mutex> call(call_mutex_);          // one job at a time, process-wide
        start_workers();
        {
            std::lock_guard<std::mutex> lk(m_);
            parts_ = &parts; device_ = device; next_ = 0; pending_ = parts.size(); failed_ = false; generation_++;
        }
        cv_work_.notify_all();
        work();
        std::unique_lock<std::mutex> lk(m_);
        cv_done_.wait(lk, [this] { return pending_ == 0; });
        parts_ = nullptr;
        return !failed_;
    }

    static HostCopyPool& instance() { static HostCopyPool* p = new HostCopyPool; return *p; }    // never destroyed: no
                                                                      // join at exit, the threads die with the process
    int threads() { start_workers(); return (int)workers_.size() + 1; }

private:
    void start_workers()
    {
        if(started_) return;
        started_ = true;
        int n = 3;
        const int hw = (int)std::thread::hardware_concurrency();
        if(hw > 0 && n > hw - 1) n = hw - 1;
        for(int k = 0; k < n; k++) workers_.emplace_back([this] { loop(); });
        for(std::thread& t : workers_) t.detach();
    }
    void loop()
    {
        unsigned long long seen = 0;
        for(;;)
        {
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_work_.wait(lk, [&] { return generation_ != seen; });
                seen = generation_;
            }
            work();
        }
    }
    void work()
    {
        int dev_set = -1;
        for(;;)
        {
            const std::vector<Part>* parts;
            size_t k;
            int dev;
            {
                std::lock_guard<std::mutex> lk(m_);
                parts = parts_;
                if(parts == nullptr || next_ >= parts->size()) return;
                k = next_++; dev = device_;
            }
            if(dev_set != dev) { cudaSetDevice(dev); dev_set = dev; }
            const Part& p = (*parts)[k];
            const bool ok = cudaEventSynchronize(p.ready) == cudaSuccess;
            if(ok) memcpy(p.dst, p.src, p.bytes);
            {
                std::lock_guard<std::mutex> lk(m_);
                if(!ok) failed_ = true;
                if(--pending_ == 0) cv_done_.notify_all();
            }
        }
    }

    std::mutex call_mutex_, m_;
    std::condition_variable cv_work_, cv_done_;
    std::vector<std::thread> workers_;
    bool started_ = false;
    const std::vector<Part>* parts_ = nullptr;
    int device_ = 0;
    size_t next_ = 0, pending_ = 0;
    bool failed_ = false;
    unsigned long long generation_ = 0;
};

bool is_pageable(const void* p)
{
    cudaPointerAttributes a{};
    if(cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeUnregistered;
}

constexpr size_t STAGE_MAX_BYTES = (size_t)256 << 20;       // larger results take the driver's path

// Device -> caller's host buffers on `st`, and waits for them.  image / ranges: destination or null; d_image /
// d_ranges: the rendered outputs (px pixels).
bool copy_results_to_host(Slot& s, char* image, float* ranges, const uint8_t* d_image, const float* d_ranges, size_t px,
                          cudaStream_t st)
{
    struct Out { char* dst; const char* src; size_t bytes; };
    Out outs[2] = { { image, (const char*)d_image, px * 3 }, { (char*)ranges, (const char*)d_ranges, px * sizeof(float) } };
    std::vector<HostCopyPool::Part> parts;
    size_t staged = 0;
    for(const Out& o : outs)
    {
        if(o.dst == nullptr) continue;
        // Page-locked destinations (cudaHostAlloc / cudaHostRegister / horizonator_host_alloc) are written by DMA at
        // PCIe speed
        if(staged + o.bytes > STAGE_MAX_BYTES || !is_pageable(o.dst))
        {
            CUDA_TRY(cudaMemcpyAsync(o.dst, o.src, o.bytes, cudaMemcpyDeviceToHost, st));
            continue;
        }
        if(s.h_stage == nullptr)
        {
            const size_t want = px * 7 < STAGE_MAX_BYTES ? px * 7 : STAGE_MAX_BYTES;
            if(cudaMallocHost(&s.h_stage, want) != cudaSuccess)
            {
                cudaGetLastError(); s.h_stage = nullptr;
                CUDA_TRY(cudaMemcpyAsync(o.dst, o.src, o.bytes, cudaMemcpyDeviceToHost, st));
                continue;
            }
            s.h_stage_bytes = want;
        }
        if(staged + o.bytes > s.h_stage_bytes)
        {
            CUDA_TRY(cudaMemcpyAsync(o.dst, o.src, o.bytes, cudaMemcpyDeviceToHost, st));
            continue;
        }
        // chunks of about 1 MB (at most ~64 per output), the last two of them cut into quarters: what remains to be
        // done after the last byte has crossed the bus is the memcpy of the last chunk
        size_t chunk = (size_t)1 << 20;
        if(o.bytes / chunk > 64) chunk = (o.bytes / 64 + 4095) & ~(size_t)4095;
        size_t n = 0;
        for(size_t off = 0; off < o.bytes; off += n)
        {
            const size_t left = o.bytes - off, want = left > 2 * chunk ? chunk : chunk / 4;
            n = left < want ? left : want;
            if(parts.size() >= s.stage_ev.size())
            {
                cudaEvent_t e;
                CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                s.stage_ev.push_back(e);
            }
            CUDA_TRY(cudaMemcpyAsync(s.h_stage + staged + off, o.src + off, n, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaEventRecord(s.stage_ev[parts.size()], st));
            parts.push_back({ o.dst + off, s.h_stage + staged + off, n, s.stage_ev[parts.size()] });
        }
        staged += o.bytes;
    }
    const bool copied = parts.empty() || HostCopyPool::instance().run(s.device, parts);
    CUDA_TRY(cudaStreamSynchronize(st));
    if(!copied)
    {
        MSG("CUDA error while the result was copied to host memory: %s", cudaGetErrorString(cudaGetLastError()));
        return false;
    }
    return true;
}

// plain asynchronous device -> host copy (the batch call: its destinations are written while later views render)
bool copy_to_host(void* dst, const void* src, size_t bytes, cudaStream_t st)
{
    CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
    return true;
}

} // namespace

extern "C" {

bool horizonator_init(horizonator_context_t* ctx,
                      float viewer_lat, float viewer_lon, float* viewer_z,
                      int offscreen_width, int offscreen_height,
                      int render_radius_cells, float render_radius_m,
                      bool use_glut, bool render_texture, bool SRTM1,
                      const char* dir_dems, const char* dir_tiles,
                      const char* tiles_name, const char* tiles_url_fmt,
                      bool allow_downloads)
{
    (void)dir_tiles; (void)tiles_name; (void)tiles_url_fmt; (void)allow_downloads;
    memset(ctx, 0, sizeof(*ctx));

    if(render_texture)
    {
        MSG("render_texture=true (OpenStreetMap texturing) is not supported by the CUDA renderer");
        return false;
    }
    if(offscreen_width > 0 && offscreen_height <= 0)
    {
        MSG("offscreen_width > 0 needs offscreen_height > 0");
        return false;
    }
    if(dir_dems == nullptr)                                             // lib:94-97
        dir_dems = SRTM1 ? "~/.horizonator/DEMs_SRTM1" : "~/.horizonator/DEMs_SRTM3";

    int ndev = 0;
    if(cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    {
        MSG("No usable CUDA device: libhorizonator renders on the GPU only (there is no CPU path)");
        return false;
    }
    int dev = 0;
    if(const char* env = getenv("HORIZONATOR_DEVICE")) dev = atoi(env);
    else if(cudaGetDevice(&dev) != cudaSuccess) dev = 0;

    if(!horizonator_dem_init(&ctx->dems, viewer_lat, viewer_lon, render_radius_cells, render_radius_m, dir_dems, SRTM1))
    {
        MSG("Couldn't init DEMs. Giving up");
        return false;
    }

    Slot* s = new Slot;
    s->device = dev;
    bool ok = false;
    do
    {
        DeviceGuard guard(dev);
        if(!guard.ok) { MSG("cudaSetDevice(%d) failed", dev); break; }
        auto fail = [](cudaError_t e, const char* what) {
            if(e != cudaSuccess) MSG("CUDA error: %s: %s", what, cudaGetErrorString(e));
            return e != cudaSuccess;
        };
        if(fail(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking), "cudaStreamCreate")) break;

        const horizonator_dem_context_t* d = &ctx->dems;
        s->cpd = d->cells_per_deg;
        s->N   = 2 * d->radius_cells;
        s->pitch = ((s->N + HZ_MESH_PAD) + 63) / 64 * 64;

        // raw tiles to the device (16 spare bytes: k_mosaic's aligned 32-bit loads may touch them)
        s->tiles.cpd = s->cpd;
        s->tiles.origin_cell[0] = d->origin_dem_cellij[0]; s->tiles.origin_cell[1] = d->origin_dem_cellij[1];
        s->tiles.ntiles[0] = d->Ndems_ij[0];               s->tiles.ntiles[1] = d->Ndems_ij[1];
        bool bad = false;
        for(int i = 0; i < d->Ndems_ij[0] && !bad; i++)
            for(int j = 0; j < d->Ndems_ij[1] && !bad; j++)
            {
                if(d->dems[i][j] == nullptr) continue;
                uint8_t* p = nullptr;
                bad = fail(cudaMalloc(&p, d->mmap_sizes[i][j] + 16), "cudaMalloc(tile)") ||
                      fail(cudaMemcpyAsync(p, d->dems[i][j], d->mmap_sizes[i][j], cudaMemcpyHostToDevice, s->stream),
                           "cudaMemcpy(tile)");
                s->tiles.tile[i][j] = p;
            }
        if(bad) break;

        // (HZ_MESH_PAD zero rows after the last: see hz_device.h)
        if(fail(cudaMalloc(&s->d_mosaic, (size_t)(s->N + HZ_MESH_PAD) * s->pitch * sizeof(int16_t)), "cudaMalloc(mosaic)")) break;
        if(fail(cudaMemsetAsync(s->d_mosaic + (size_t)s->N * s->pitch, 0, (size_t)HZ_MESH_PAD * s->pitch * sizeof(int16_t), s->stream),
                "cudaMemset(mosaic)")) break;
        s->nb = (s->N - 1 + HZ_BLOCK_CELLS - 1) / HZ_BLOCK_CELLS;
        s->nt = (s->N - 1 + HZ_TILE_CELLS - 1) / HZ_TILE_CELLS;
        if(fail(cudaMalloc(&s->d_mm_block, (size_t)s->nb * s->nb * sizeof(short2)), "cudaMalloc(pyramid)")) break;
        if(fail(cudaMalloc(&s->d_mm_tile, (size_t)s->nt * s->nt * sizeof(short2)), "cudaMalloc(pyramid)")) break;
        if(!alloc_set(s->main, 1, false) || ensure_views(*s, s->main, 1) != 1) break;
        if(fail(hz_launch_mosaic(s->tiles, s->d_mosaic, s->N, s->pitch, s->stream), "k_mosaic")) break;
        if(fail(hz_launch_pyramid(s->d_mosaic, s->N, s->pitch, s->d_mm_block, s->nb, s->d_mm_tile, s->nt, s->stream),
                "k_minmax")) break;

        // without an offscreen size the reference opens a 1024x1024 window (lib:142)
        const int W = offscreen_width > 0 ? offscreen_width : 1024;
        const int H = offscreen_width > 0 ? offscreen_height : 1024;
        if(!alloc_target(*s, W, H)) break;
        if(fail(cudaStreamSynchronize(s->stream), "DEM upload/decode")) break;
        ok = true;
    } while(0);

    if(!ok)
    {
        destroy_slot(s);
        horizonator_dem_deinit(&ctx->dems);
        memset(ctx, 0, sizeof(*ctx));
        return false;
    }

    {
        std::lock_guard<std::mutex> lock(g_table_mutex);
        size_t k = 0;
        while(k < g_table.size() && g_table[k] != nullptr) k++;
        if(k == g_table.size()) g_table.push_back(s); else g_table[k] = s;
        ctx->program = (uint32_t)(k + 1);
    }

    const int n1 = 2 * ctx->dems.radius_cells - 1;
    ctx->Ntriangles     = n1 * n1 * 2;                                  // lib:202-203
    ctx->render_texture = false;
    ctx->use_glut       = use_glut;
    ctx->glut_window    = 1;
    // the 17 GL uniform locations of the reference: no meaning here, -1 = "no such uniform"
    memset(&ctx->uniform_aspect, 0xFF,
           offsetof(horizonator_context_t, uniform_zfar_color) + sizeof(int32_t) - offsetof(horizonator_context_t, uniform_aspect));
    if(offscreen_width > 0)
    {
        ctx->offscreen.inited = true;
        ctx->offscreen.width  = offscreen_width;
        ctx->offscreen.height = offscreen_height;
    }

    horizonator_move(ctx, viewer_z, viewer_lat, viewer_lon);           // lib:611
    horizonator_set_zextents(ctx, HORIZONATOR_ZNEAR_DEFAULT, HORIZONATOR_ZFAR_DEFAULT,
                             HORIZONATOR_ZNEAR_DEFAULT, HORIZONATOR_ZFAR_DEFAULT);
    horizonator_pan_zoom(ctx, -45.f, 45.f);                             // lib:670
    return true;
}

void horizonator_deinit(horizonator_context_t* ctx)
{
    if(ctx == nullptr) return;
    Slot* s = nullptr;
    if(ctx->Ntriangles > 0 && ctx->program != 0)
    {
        std::lock_guard<std::mutex> lock(g_table_mutex);
        if(ctx->program <= g_table.size())
        {
            s = g_table[ctx->program - 1];
            g_table[ctx->program - 1] = nullptr;
        }
    }
    destroy_slot(s);
    if(ctx->Ntriangles > 0) horizonator_dem_deinit(&ctx->dems);
    ctx->Ntriangles  = 0;
    ctx->program     = 0;
    ctx->glut_window = 0;
    ctx->offscreen.inited = false;
}

bool horizonator_resized(const horizonator_context_t* ctx, int width, int height)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    if(ctx->offscreen.inited)
    {
        MSG("Resizing an offscreen context is not supported");          // the reference asserts here
        return false;
    }
    if(width <= 0 || height <= 0) return false;
    DeviceGuard g(s->device);
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return alloc_target(*s, width, height);
}

bool horizonator_pan_zoom(const horizonator_context_t* ctx, float az_deg0, float az_deg1)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    s->view.az_deg0 = az_deg0;      // stored as given, like the uniforms at lib:833-834
    s->view.az_deg1 = az_deg1;
    return true;
}

bool horizonator_move(horizonator_context_t* ctx, float* viewer_z, float viewer_lat, float viewer_lon)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    const float az0 = s->view.az_deg0, az1 = s->view.az_deg1;
    if(!compute_move(ctx, viewer_z, viewer_lat, viewer_lon, s->view)) return false;
    s->view.az_deg0 = az0; s->view.az_deg1 = az1;
    ctx->viewer_lat = viewer_lat;                                       // lib:812-813
    ctx->viewer_lon = viewer_lon;
    return true;
}

bool horizonator_set_zextents(horizonator_context_t* ctx,
                              float znear, float zfar, float znear_color, float zfar_color)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    if(!(znear > 0.0f && znear_color > 0.0f && zfar > 0.0f && zfar_color > 0.0f)) return false;   // lib:875-877
    s->znear = znear; s->zfar = zfar; s->znear_color = znear_color; s->zfar_color = zfar_color;
    return true;
}

bool horizonator_redraw(const horizonator_context_t* ctx)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    DeviceGuard g(s->device);
    if(!enqueue_render(*s, s->view, 0, s->W, single_out(s->d_image, s->d_ranges), s->stream)) return false;
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return true;
}

bool horizonator_render_offscreen(const horizonator_context_t* ctx, char* image, float* ranges)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    if(!ctx->offscreen.inited)
    {
        MSG("Prior to calling horizonator_render_offscreen(), the context must have been inited for offscreen rendering with horizonator_init(offscreen_width,height > 0)");
        return false;
    }
    DeviceGuard g(s->device);
    const size_t px = (size_t)s->W * s->H;
    if(!enqueue_render(*s, s->view, 0, s->W,
                       single_out(image ? s->d_image : nullptr, ranges ? s->d_ranges : nullptr), s->stream)) return false;
    return copy_results_to_host(*s, image, ranges, s->d_image, s->d_ranges, px, s->stream);
}

bool horizonator_pick(const horizonator_context_t* ctx, float* lat, float* lon, int x, int y)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || !s->have_render) return false;
    if(x < 0 || y < 0 || x >= s->W || y >= s->H) return false;
    DeviceGuard g(s->device);
    unsigned long long key = 0;
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    CUDA_TRY(cudaMemcpy(&key, s->main.sc[0].d_vis + (size_t)(s->H - 1 - y) * s->W + x, sizeof(key), cudaMemcpyDeviceToHost));
    const float depth = (float)((double)hz_key_q(key, s->main.sc[0].last_epoch) * (1.0 / 16777215.0));
    if(depth >= 1.0f) return false;                                     // lib:1272
    // lib:1282-1295: the depth is treated as horizontal distance
    const double range_en = depth * (s->zfar - s->znear) + s->znear;
    return horizonator_unproject(lat, lon, x, y, -1., range_en,
                                 ctx->viewer_lat, s->view.cos_viewer_lat, ctx->viewer_lon,
                                 s->view.az_deg0, s->view.az_deg1, s->W, s->H);
}

// ---- pure host geometry (lib:1053-1213): double precision, no device involved ----------------------------

static double unwrap_near_rad_d(double x, double near)
{
    const double d = (x - near) / (2. * M_PI);
    return (d - round(d)) * 2. * M_PI + near;
}

bool horizonator_x_from_az(double* x, double* az_ndc_per_rad,
                           double az_rad, double az_rad0, double az_rad1, int width)
{
    az_rad1 = unwrap_near_rad_d(az_rad1 - az_rad0, M_PI) + az_rad0;
    const double center = (az_rad0 + az_rad1) / 2.;
    az_rad = unwrap_near_rad_d(az_rad, center);
    const double per_rad = 2.0 / (az_rad1 - az_rad0);
    const double az_ndc  = (az_rad - center) * per_rad;
    if(!(-1. <= az_ndc && az_ndc <= 1.)) return false;
    if(az_ndc_per_rad != nullptr) *az_ndc_per_rad = per_rad;
    *x = (az_ndc + 1.) / 2. * width - 0.5;                               // NDC [-1,1] -> pixel (-0.5, W-0.5)
    return true;
}

bool horizonator_project(double* x, double* y, double* range,
                         double lat_viewer, double cos_lat_viewer, double lon_viewer, double ele_viewer,
                         double lat, double lon, double ele,
                         double az_rad0, double az_rad1, int width, int height)
{
    const float Rearth = 6371000.0;
    const double dlat = (lat - lat_viewer) * M_PI / 180;
    const double dlon = (lon - lon_viewer) * M_PI / 180;
    const double east  = dlon * Rearth * cos_lat_viewer;
    const double north = dlat * Rearth;
    const double d2 = east * east + north * north;

    double per_rad;
    if(!horizonator_x_from_az(x, &per_rad, atan2(east, north), az_rad0, az_rad1, width)) return false;

    const double h = ele - ele_viewer;
    *range = sqrt(d2 + h * h);
    const double aspect = (double)width / (double)height;
    const double el_ndc = atan2(h, sqrt(d2)) * aspect * per_rad;
    if(!(-1. <= el_ndc && el_ndc <= 1.)) return false;
    *y = (-el_ndc + 1.) / 2. * height - 0.5;
    return true;
}

bool horizonator_unproject(float* lat, float* lon, int x, int y,
                           double range_enh, double range_en,
                           double lat_viewer, double cos_lat_viewer, double lon_viewer,
                           double az_deg0, double az_deg1, int width, int height)
{
    if(1 != (range_enh > 0.) + (range_en > 0.)) return false;
    const float Rearth = 6371000.0;
    // mixed float/double exactly as lib:1185-1186
    const float az_ndc = ((float)x + 0.5f) / (float)width * 2.f - 1.f;
    const float az     = (az_ndc * (az_deg1 - az_deg0) / 2.f + (az_deg1 + az_deg0) / 2.f) * M_PI / 180.0f;
    if(range_en <= 0)
    {
        const double aspect = (double)width / (double)height;
        const double el_ndc = ((double)y + 0.5) / (double)height * 2. - 1.;
        const double el     = el_ndc * (az_deg1 - az_deg0) / 2. / aspect * M_PI / 180.0;
        range_en = cos(el) * range_enh;
    }
    const float e = range_en * sinf(az);
    const float n = range_en * cosf(az);
    *lon = lon_viewer + e / Rearth / M_PI * 180. / cos_lat_viewer;
    *lat = lat_viewer + n / Rearth / M_PI * 180.;
    return true;
}

// ---- additive API (include/horizonator-batch.h) -----------------------------------------------------------

// Common part of the two batch calls.  The views are cut into chunks of up to VIEWS_PER_SET; a chunk is rendered by
// ONE chain of kernel launches whose grids have a view dimension (one parameter copy and one CUDA-graph launch per
// chunk, whatever its size), on the stream of one of up to N_SETS_MAX view sets, so that the tails of one chunk's
// kernels overlap another chunk's.  The sets start after everything already queued on `st`, and `st` continues after
// all of them.  to_host: outputs go through the views' device staging buffers and device->host copies on the set's
// stream, which overlap the other sets' kernels.
static bool render_batch_common(const horizonator_context_t* ctx, Slot* s, int n, const horizonator_view_t* views,
                                uint8_t* images, float* ranges, bool to_host, cudaStream_t st)
{
    const size_t px = (size_t)s->W * s->H;
    std::vector<ViewState> vs((size_t)n);
    for(int k = 0; k < n; k++)
    {
        float z = views[k].viewer_z;
        if(!compute_move(ctx, &z, views[k].lat, views[k].lon, vs[k])) return false;
        vs[k].az_deg0 = views[k].az_deg0; vs[k].az_deg1 = views[k].az_deg1;
    }
    if(n == 0) return true;

    // chunk size: the views spread evenly over the sets, at most VIEWS_PER_SET each, at most what fits in memory
    int n_sets = 0, chunk = 0;
    if(n > 1)
    {
        // (no fewer than 8 to a chunk where there are that many: a launch pays off with views to share it)
        n_sets = N_SETS_MAX;
        chunk = (n + n_sets - 1) / n_sets;
        if(chunk < 8) chunk = n < 8 ? n : 8;
        if(chunk > VIEWS_PER_SET) chunk = VIEWS_PER_SET;
        n_sets = (n + chunk - 1) / chunk < n_sets ? (n + chunk - 1) / chunk : n_sets;
        for(int g = 0; g < n_sets; g++)
        {
            ViewSet* set = batch_set(*s, g);
            const int have = set ? ensure_views(*s, *set, chunk) : 0;
            if(have < chunk)
            {
                if(g == 0) chunk = have;              // every set gets what the first one could have
                else       n_sets = g;                // later sets: do without them
                if(chunk < 1) { n_sets = 0; break; }
            }
        }
    }

    if(n_sets == 0)
    {
        // one view, or no memory for a set: one at a time on the context's own scratch
        for(int k = 0; k < n; k++)
        {
            uint8_t* di = images ? (to_host ? s->d_image  : images + (size_t)k * px * 3) : nullptr;
            float*   dr = ranges ? (to_host ? s->d_ranges : ranges + (size_t)k * px)     : nullptr;
            if(!enqueue_render(*s, vs[k], 0, s->W, single_out(di, dr), st)) return false;
            if(to_host)
            {
                if(images && !copy_to_host(images + (size_t)k * px * 3, di, px * 3, st)) return false;
                if(ranges && !copy_to_host(ranges + (size_t)k * px, dr, px * sizeof(float), st)) return false;
            }
        }
        s->have_render = false;     // the visibility buffer no longer matches the context's own view
        return true;
    }

    CUDA_TRY(cudaEventRecord(s->fork_ev, st));
    for(int g = 0; g < n_sets; g++) CUDA_TRY(cudaStreamWaitEvent(s->sets[g]->stream, s->fork_ev, 0));
    bool ok = true;
    std::vector<OutSpec> outs((size_t)chunk);
    for(int k0 = 0, c = 0; k0 < n && ok; k0 += chunk, c++)
    {
        ViewSet& set = *s->sets[c % n_sets];
        const int m = n - k0 < chunk ? n - k0 : chunk;
        for(int k = 0; k < m; k++)
            outs[k] = single_out(images ? (to_host ? set.sc[k].d_image  : images + (size_t)(k0 + k) * px * 3) : nullptr,
                                 ranges ? (to_host ? set.sc[k].d_ranges : ranges + (size_t)(k0 + k) * px)     : nullptr);
        ok = enqueue_views(*s, set, m, &vs[k0], 0, s->W, outs.data(), set.stream);
        for(int k = 0; k < m && ok && to_host; k++)
        {
            if(images) ok = ok && copy_to_host(images + (size_t)(k0 + k) * px * 3, set.sc[k].d_image, px * 3, set.stream);
            if(ranges) ok = ok && copy_to_host(ranges + (size_t)(k0 + k) * px, set.sc[k].d_ranges, px * sizeof(float), set.stream);
        }
    }
    if(!ok)
    {
        // whatever was queued may still be writing into the caller's buffers: let it finish before reporting failure
        for(int g = 0; g < n_sets; g++) cudaStreamSynchronize(s->sets[g]->stream);
        cudaGetLastError();
        return false;
    }
    for(int g = 0; g < n_sets; g++)
    {
        CUDA_TRY(cudaEventRecord(s->sets[g]->done, s->sets[g]->stream));
        CUDA_TRY(cudaStreamWaitEvent(st, s->sets[g]->done, 0));
    }
    return true;
}

// ---- viewsheds (horizonator-batch.h) -------------------------------------------------------------------------------
//
// The views go in chunks of up to HZ_VS_MAX_VIEWS, each one k_viewshed launch (gridDim.y = view) into its masks --
// the caller's, or the scratch when the masks are not wanted in device memory -- then k_viewshed_count into the
// counts and/or a copy of the masks to host memory, all on `st`.
static bool viewshed_common(const horizonator_context_t* ctx, Slot* s, int n, const horizonator_view_t* views,
                            float target_height, uint32_t* d_masks, uint32_t* d_counts, uint32_t* h_masks,
                            cudaStream_t st)
{
    const int N = s->N, w32 = (N + 31) / 32;
    const size_t mwords = (size_t)N * w32;
    std::vector<HzViewshedEye> eyes((size_t)n);
    for(int k = 0; k < n; k++)
    {
        ViewState vs;
        float z = views[k].viewer_z;
        if(!compute_move(ctx, &z, views[k].lat, views[k].lon, vs)) return false;
        if(!(vs.viewer_cell_i >= 0.f && vs.viewer_cell_i < (float)(N - 1) &&
             vs.viewer_cell_j >= 0.f && vs.viewer_cell_j < (float)(N - 1)))
        {
            MSG("viewshed: the eye of view %d (cell %g, %g) is not inside the loaded square [0, %d)", k,
                (double)vs.viewer_cell_i, (double)vs.viewer_cell_j, N - 1);
            return false;
        }
        eyes[k] = HzViewshedEye{ vs.viewer_cell_i, vs.viewer_cell_j, vs.viewer_z, vs.cos_viewer_lat };
    }
    if(n == 0) return true;

    const int chunk = n < HZ_VS_MAX_VIEWS ? n : HZ_VS_MAX_VIEWS;
    if(s->vs_done == nullptr) CUDA_TRY(cudaEventCreateWithFlags(&s->vs_done, cudaEventDisableTiming));
    else CUDA_TRY(cudaStreamWaitEvent(st, s->vs_done, 0));
    if(d_masks == nullptr && s->vs_mask_views < chunk)
    {
        CUDA_TRY(cudaEventSynchronize(s->vs_done));
        cudaFree(s->d_vs_masks);
        s->d_vs_masks = nullptr; s->vs_mask_views = 0;
        if(cudaMalloc(&s->d_vs_masks, (size_t)chunk * mwords * sizeof(uint32_t)) != cudaSuccess)
        {
            cudaGetLastError();
            MSG("Could not allocate the viewshed masks of %d views (%zu MB)", chunk, (size_t)chunk * mwords * 4 >> 20);
            return false;
        }
        s->vs_mask_views = chunk;
    }

    HzViewshed p{};
    p.mosaic = s->d_mosaic; p.N = N; p.pitch = s->pitch; p.w32 = w32;
    p.deg_per_cell = 1.0f / (float)s->cpd;                                // lib:577
    p.curvature = s->curvature;
    p.target_height = target_height;
    for(int k0 = 0; k0 < n; k0 += chunk)
    {
        const int m = n - k0 < chunk ? n - k0 : chunk;
        p.masks = d_masks ? d_masks + (size_t)k0 * mwords : s->d_vs_masks;
        for(int k = 0; k < m; k++) p.eye[k] = eyes[(size_t)(k0 + k)];
        CUDA_TRY(cudaMemsetAsync(p.masks, 0, (size_t)m * mwords * sizeof(uint32_t), st));
        CUDA_TRY(hz_launch_viewshed(p, m, st));
        if(d_counts) CUDA_TRY(hz_launch_viewshed_count(p.masks, m, N, w32, d_counts, st));
        if(h_masks)
            CUDA_TRY(cudaMemcpyAsync(h_masks + (size_t)k0 * mwords, p.masks, (size_t)m * mwords * sizeof(uint32_t),
                                     cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(cudaEventRecord(s->vs_done, st));
    return true;
}

bool horizonator_viewshed_device(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                                 float target_height_m, void* d_masks, void* d_counts, void* stream)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || n < 0 || (n > 0 && views == nullptr)) return false;
    if(d_masks == nullptr && d_counts == nullptr)
    {
        MSG("horizonator_viewshed_device: neither masks nor counts asked for");
        return false;
    }
    DeviceGuard g(s->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if(!viewshed_common(ctx, s, n, views, target_height_m, (uint32_t*)d_masks, (uint32_t*)d_counts, nullptr, st))
        return false;
    if(stream == nullptr) CUDA_TRY(cudaStreamSynchronize(st));
    return true;
}

bool horizonator_viewshed(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                          float target_height_m, uint32_t* masks, uint32_t* counts)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || n < 0 || (n > 0 && views == nullptr)) return false;
    if(masks == nullptr && counts == nullptr)
    {
        MSG("horizonator_viewshed: neither masks nor counts asked for");
        return false;
    }
    DeviceGuard g(s->device);
    const size_t cells = (size_t)s->N * s->N;
    if(counts && n > 0 && s->d_vs_counts == nullptr)
    {
        if(s->vs_done) CUDA_TRY(cudaEventSynchronize(s->vs_done));
        if(cudaMalloc(&s->d_vs_counts, cells * sizeof(uint32_t)) != cudaSuccess)
        {
            cudaGetLastError();
            MSG("Could not allocate the viewshed counts (%zu MB)", cells * 4 >> 20);
            return false;
        }
    }
    // the counts' upload waits for whatever an earlier call still does with the same buffer
    if(counts && n > 0 && s->vs_done) CUDA_TRY(cudaStreamWaitEvent(s->stream, s->vs_done, 0));
    if(counts && n > 0) CUDA_TRY(cudaMemcpyAsync(s->d_vs_counts, counts, cells * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
    if(!viewshed_common(ctx, s, n, views, target_height_m, nullptr, counts ? s->d_vs_counts : nullptr, masks, s->stream))
    {
        cudaStreamSynchronize(s->stream);
        cudaGetLastError();
        return false;
    }
    if(counts && n > 0) CUDA_TRY(cudaMemcpyAsync(counts, s->d_vs_counts, cells * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return true;
}

bool horizonator_render_batch_device(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                                     void* d_images, void* d_ranges, void* stream)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || n < 0 || (n > 0 && views == nullptr)) return false;
    DeviceGuard g(s->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if(!render_batch_common(ctx, s, n, views, (uint8_t*)d_images, (float*)d_ranges, false, st)) return false;
    if(stream == nullptr) CUDA_TRY(cudaStreamSynchronize(st));
    return true;
}

bool horizonator_render_batch(const horizonator_context_t* ctx, int n, const horizonator_view_t* views,
                              char* images, float* ranges)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || n < 0 || (n > 0 && views == nullptr)) return false;
    DeviceGuard g(s->device);
    if(!render_batch_common(ctx, s, n, views, (uint8_t*)images, ranges, true, s->stream)) return false;
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return true;
}

bool horizonator_render_wedge_device(const horizonator_context_t* ctx, int x0, int x1,
                                     void* d_image, void* d_ranges, void* stream)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    if(x0 < 0 || x1 > s->W || x0 >= x1)
    {
        MSG("wedge columns [%d,%d) are not inside [0,%d)", x0, x1, s->W);
        return false;
    }
    DeviceGuard g(s->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if(!enqueue_render(*s, s->view, x0, x1, single_out((uint8_t*)d_image, (float*)d_ranges), st)) return false;
    if(stream == nullptr) CUDA_TRY(cudaStreamSynchronize(st));
    return true;
}

bool horizonator_render_wedge_host(const horizonator_context_t* ctx, int x0, int x1, char* image, float* ranges)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    if(x0 < 0 || x1 > s->W || x0 >= x1)
    {
        MSG("wedge columns [%d,%d) are not inside [0,%d)", x0, x1, s->W);
        return false;
    }
    if(image == nullptr && ranges == nullptr) return true;
    DeviceGuard g(s->device);
    cudaStream_t st = s->stream;
    // the context's own output buffers serve as the slab [H][x1-x0]; from there straight into the caller's columns
    const size_t w = (size_t)(x1 - x0);
    if(!enqueue_render(*s, s->view, x0, x1, single_out(image ? s->d_image : nullptr, ranges ? s->d_ranges : nullptr), st)) return false;
    if(image)  CUDA_TRY(cudaMemcpy2DAsync(image + (size_t)x0 * 3, (size_t)s->W * 3, s->d_image, w * 3, w * 3, (size_t)s->H,
                                          cudaMemcpyDeviceToHost, st));
    if(ranges) CUDA_TRY(cudaMemcpy2DAsync(ranges + x0, (size_t)s->W * sizeof(float), s->d_ranges, w * sizeof(float),
                                          w * sizeof(float), (size_t)s->H, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return true;
}

bool horizonator_host_register(void* p, size_t bytes)
{
    if(p == nullptr || bytes == 0) return false;
    const cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
    if(e != cudaSuccess)
    {
        MSG("cudaHostRegister(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
        cudaGetLastError();
        return false;
    }
    return true;
}

bool horizonator_host_unregister(void* p)
{
    if(p == nullptr) return false;
    if(cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return false; }
    return true;
}

// ---- wedge-sharded panoramas assembled over NVLink ---------------------------------------------------------

bool horizonator_peer_alloc(const horizonator_context_t* ctx, size_t bytes, void** d_ptr, unsigned char handle[64])
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || d_ptr == nullptr || handle == nullptr || bytes == 0) return false;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    DeviceGuard g(s->device);
    void* p = nullptr;
    CUDA_TRY(cudaMalloc(&p, bytes));
    cudaIpcMemHandle_t h;
    const cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if(e != cudaSuccess)
    {
        MSG("cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
        cudaFree(p);
        return false;
    }
    memcpy(handle, &h, 64);
    *d_ptr = p;
    return true;
}

bool horizonator_peer_open(const horizonator_context_t* ctx, const unsigned char handle[64], void** d_ptr)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || d_ptr == nullptr || handle == nullptr) return false;
    DeviceGuard g(s->device);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CUDA_TRY(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return true;
}

bool horizonator_peer_close(const horizonator_context_t* ctx, void* d_ptr)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || d_ptr == nullptr) return false;
    DeviceGuard g(s->device);
    CUDA_TRY(cudaIpcCloseMemHandle(d_ptr));
    return true;
}

bool horizonator_peer_free(const horizonator_context_t* ctx, void* d_ptr)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    DeviceGuard g(s->device);
    CUDA_TRY(cudaFree(d_ptr));
    return true;
}

bool horizonator_render_wedge_peers(const horizonator_context_t* ctx, int x0, int x1, int n_peers,
                                    void* const* d_images, void* const* d_ranges, void* stream)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    if(x0 < 0 || x1 > s->W || x0 >= x1)
    {
        MSG("wedge columns [%d,%d) are not inside [0,%d)", x0, x1, s->W);
        return false;
    }
    if(n_peers < 1 || n_peers > HZ_MAX_OUT || (d_images == nullptr && d_ranges == nullptr))
    {
        MSG("need 1..%d destinations and at least one kind of output", HZ_MAX_OUT);
        return false;
    }
    OutSpec out;
    out.n = n_peers; out.stride = s->W; out.x_off = x0;
    for(int d = 0; d < n_peers; d++)
    {
        out.image[d]  = d_images ? (uint8_t*)d_images[d] : nullptr;
        out.ranges[d] = d_ranges ? (float*)d_ranges[d]   : nullptr;
        if((d_images && out.image[d] == nullptr) || (d_ranges && out.ranges[d] == nullptr))
        {
            MSG("destination %d is null", d);
            return false;
        }
    }
    DeviceGuard g(s->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if(!enqueue_render(*s, s->view, x0, x1, out, st)) return false;
    if(stream == nullptr) CUDA_TRY(cudaStreamSynchronize(st));
    return true;
}

bool horizonator_peer_barrier(const horizonator_context_t* ctx, int n_ranks, int rank, void* const* d_flags,
                              unsigned int epoch, void* stream)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || d_flags == nullptr || n_ranks < 1 || n_ranks > HZ_MAX_OUT || rank < 0 || rank >= n_ranks) return false;
    HzPeerFlags f{};
    f.n = n_ranks; f.rank = rank;
    for(int r = 0; r < n_ranks; r++)
    {
        if(d_flags[r] == nullptr) return false;
        f.arrive[r] = (uint32_t*)d_flags[r];
    }
    DeviceGuard g(s->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    CUDA_TRY(hz_launch_peer_barrier(f, epoch, st));
    if(stream == nullptr) CUDA_TRY(cudaStreamSynchronize(st));
    return true;
}

bool horizonator_set_seam_wrap(const horizonator_context_t* ctx, bool on)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    s->seam_wrap = on;
    return true;
}

bool horizonator_set_lod(const horizonator_context_t* ctx, float max_cell_pixels)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    if(!(max_cell_pixels >= 0.f))
    {
        MSG("max_cell_pixels %g is negative", (double)max_cell_pixels);
        return false;
    }
    if((max_cell_pixels > 0.f) != (s->lod_pixels > 0.f))
    {
        // the captured chains launch a different instantiation of k_blocks: wait for what is in flight, drop them
        DeviceGuard g(s->device);
        CUDA_TRY(cudaStreamSynchronize(s->stream));
        for(ViewSet* v : s->sets) CUDA_TRY(cudaStreamSynchronize(v->stream));
        if(s->main.busy_recorded) CUDA_TRY(cudaEventSynchronize(s->main.busy));
        for(ViewSet* v : s->sets) if(v->busy_recorded) CUDA_TRY(cudaEventSynchronize(v->busy));
        drop_graphs(s->main);
        for(ViewSet* v : s->sets) drop_graphs(*v);
    }
    s->lod_pixels = max_cell_pixels;
    return true;
}

bool horizonator_set_earth_curvature(const horizonator_context_t* ctx, bool on, float refraction)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    if(on && !(refraction >= 0.f && refraction < 1.f))
    {
        MSG("refraction coefficient %g is not in [0,1)", (double)refraction);
        return false;
    }
    s->curvature = on ? (1.0f - refraction) / (2.0f * 6371000.0f) : 0.0f;
    return true;
}

bool horizonator_debug_device_math(int n, const float* e, const float* north, const float* h, const float* d2,
                                   float* az, float* el)
{
    if(n < 0 || (n > 0 && (!e || !north || !h || !d2 || !az || !el))) return false;
    if(n == 0) return true;
    float* d = nullptr;
    const size_t bytes = (size_t)n * sizeof(float);
    CUDA_TRY(cudaMalloc(&d, 6 * bytes));
    bool ok = cudaMemcpy(d, e, bytes, cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemcpy(d + n, north, bytes, cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemcpy(d + 2 * (size_t)n, h, bytes, cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemcpy(d + 3 * (size_t)n, d2, bytes, cudaMemcpyHostToDevice) == cudaSuccess &&
              hz_launch_math_probe(n, d, d + n, d + 2 * (size_t)n, d + 3 * (size_t)n, d + 4 * (size_t)n, d + 5 * (size_t)n, nullptr) == cudaSuccess &&
              cudaMemcpy(az, d + 4 * (size_t)n, bytes, cudaMemcpyDeviceToHost) == cudaSuccess &&
              cudaMemcpy(el, d + 5 * (size_t)n, bytes, cudaMemcpyDeviceToHost) == cudaSuccess;
    if(!ok) MSG("CUDA error in horizonator_debug_device_math: %s", cudaGetErrorString(cudaGetLastError()));
    cudaFree(d);
    return ok;
}

void* horizonator_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if(cudaMallocHost(&p, bytes) != cudaSuccess)
    {
        MSG("cudaMallocHost(%zu) failed", bytes);
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void horizonator_host_free(void* p)
{
    if(p != nullptr) cudaFreeHost(p);
}

bool horizonator_download_mosaic(const horizonator_context_t* ctx, int16_t* mosaic)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || mosaic == nullptr) return false;
    DeviceGuard g(s->device);
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    CUDA_TRY(cudaMemcpy2D(mosaic, (size_t)s->N * sizeof(int16_t), s->d_mosaic, (size_t)s->pitch * sizeof(int16_t),
                          (size_t)s->N * sizeof(int16_t), s->N, cudaMemcpyDeviceToHost));
    return true;
}

bool horizonator_time_mosaic(const horizonator_context_t* ctx, int reps, float* ms_per_run)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || reps <= 0 || ms_per_run == nullptr) return false;
    DeviceGuard g(s->device);
    cudaEvent_t a, b;
    CUDA_TRY(cudaEventCreate(&a));
    CUDA_TRY(cudaEventCreate(&b));
    CUDA_TRY(hz_launch_mosaic(s->tiles, s->d_mosaic, s->N, s->pitch, s->stream));      // warm-up
    CUDA_TRY(cudaEventRecord(a, s->stream));
    for(int k = 0; k < reps; k++) CUDA_TRY(hz_launch_mosaic(s->tiles, s->d_mosaic, s->N, s->pitch, s->stream));
    CUDA_TRY(cudaEventRecord(b, s->stream));
    CUDA_TRY(cudaEventSynchronize(b));
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a); cudaEventDestroy(b);
    *ms_per_run = ms / (float)reps;
    return true;
}

bool horizonator_profile_enable(const horizonator_context_t* ctx, bool on)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    s->profiling = on;
    s->collect_stats = on;
    return true;
}

bool horizonator_profile_read(const horizonator_context_t* ctx, float out_ms[6], int* renders)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || out_ms == nullptr || renders == nullptr) return false;
    DeviceGuard g(s->device);
    double sum[PROF_EVENTS - 1] = {};
    const size_t n = s->prof_used / PROF_EVENTS;
    for(size_t r = 0; r < n; r++)
    {
        cudaEvent_t* ev = &s->prof_events[PROF_EVENTS * r];
        CUDA_TRY(cudaEventSynchronize(ev[PROF_EVENTS - 1]));
        for(int k = 0; k < PROF_EVENTS - 1; k++)
        {
            float ms = 0;
            CUDA_TRY(cudaEventElapsedTime(&ms, ev[k], ev[k + 1]));
            sum[k] += ms;
        }
    }
    for(int k = 0; k < PROF_EVENTS - 1; k++) out_ms[k] = n ? (float)(sum[k] / (double)n) : 0.f;
    *renders = (int)n;
    s->prof_used = 0;
    return true;
}

bool horizonator_last_render_stats(const horizonator_context_t* ctx, unsigned int out[5])
{
    Slot* s = slot_of(ctx);
    if(s == nullptr) return false;
    DeviceGuard g(s->device);
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    unsigned int counters[N_COUNTERS] = {};
    CUDA_TRY(cudaMemcpy(counters, s->main.sc[0].d_counters, sizeof(counters), cudaMemcpyDeviceToHost));
    out[0] = counters[0];
    for(int b = 0; b < MAX_BANDS; b++) out[0] += counters[7 + 4 * b];
    out[1] = 2 * s->big_capacity; out[2] = s->launches_last; out[3] = (unsigned)s->device;
    out[4] = counters[2];
    for(int b = 0; b < MAX_BANDS; b++) out[4] += counters[6 + 4 * b];     // triangle lists of the near pass and the bands
    return true;
}

bool horizonator_render_counters(const horizonator_context_t* ctx, unsigned int out[16])
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || out == nullptr) return false;
    DeviceGuard g(s->device);
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    CUDA_TRY(cudaMemcpy(out, s->main.sc[0].d_counters + STATS_AT, HZ_STAT_COUNT * sizeof(unsigned int), cudaMemcpyDeviceToHost));
    return true;
}

bool horizonator_horizon_profile_device(const horizonator_context_t* ctx, const void* d_ranges, int n,
                                        void* d_rows, void* d_range, void* stream)
{
    Slot* s = slot_of(ctx);
    if(s == nullptr || n < 0 || d_ranges == nullptr || d_rows == nullptr || d_range == nullptr) return false;
    DeviceGuard g(s->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    CUDA_TRY(hz_launch_horizon((const float*)d_ranges, n, s->W, s->H, (int*)d_rows, (float*)d_range, st));
    if(stream == nullptr) CUDA_TRY(cudaStreamSynchronize(st));
    return true;
}

} // extern "C"
