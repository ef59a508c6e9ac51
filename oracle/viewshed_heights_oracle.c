/* viewshed_heights_oracle.c -- TEST INFRASTRUCTURE (oracle).  Not part of the product; only tests/ and tools may use it.
 *
 *   vs_oracle_r2_heights  the heights of the R2 walk (include/horizonator-batch.h, horizonator_viewshed_heights): per
 *                         vertex of the oracle context's DEM square the least height above the ground at which some
 *                         ray of the current eye sees it -- the GPU kernel (k_viewshed_heights) must match it bit for
 *                         bit
 *
 * The scene, the eye, the targets, the heights and the metres are viewshed_oracle.c's own, included below so that
 * they exist once; vs_ray_heights() is vs_ray() line for line, with the mask's test q >= smax replaced by the step's
 * height.  heights: N x N float, row j north, column i east; overwritten.  Returns false (heights untouched) when
 * the eye is not inside [0, N-1)^2.
 *
 * Build with -ffp-contract=off, like the rest of oracle/: one IEEE rounding per source operator.
 */
#include "viewshed_oracle.c"

/* heights[j][i] = min(heights[j][i], e) for e >= +0 or +inf: the minimum of the 32-bit patterns, which order like the
   floats there, by compare-and-swap -- exact and independent of the order the threads come in */
static void vs_min(float* heights, int N, int i, int j, float e)
{
    uint32_t* h = (uint32_t*)(heights + (size_t)j * N + i);
    uint32_t v;
    memcpy(&v, &e, sizeof v);
    uint32_t cur = __atomic_load_n(h, __ATOMIC_RELAXED);
    while(v < cur && !__atomic_compare_exchange_n(h, &cur, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
}

/* One ray of R2, as vs_ray(): the height e = smax * D - A of each step, with A the decided vertex's apparent height
   and D its horizontal distance (the terms of vs_ray's q before the target height), folded into `heights` */
static void vs_ray_heights(const vs_scene_t* s, int ti, int tj, float* heights)
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
        /* the vertex this step decides: (a, rint(b)), its apparent height A at distance D against the steps before
           it; -inf (the first step), negatives, -0 and NaN all become +0 */
        const float zr = r == b0 ? z0 : z1;
        const float mr = vs_metres((float)r, vb, dpc, sb);
        const float d2r = ma * ma + mr * mr;
        const float A = zr - vz - curv * d2r;
        const float e = smax * sqrtf(d2r) - A;
        vs_min(heights, N, xmaj ? a : r, xmaj ? r : a, e > 0.f ? e : 0.f);
        smax = sl > smax ? sl : smax;
        if(a == ta) break;
    }
}

bool vs_oracle_r2_heights(const oracle_context_t* ctx, const int16_t* z, float curvature, int nthreads, float* heights)
{
    vs_scene_t s;
    if(!vs_scene(ctx, z, curvature, &s)) return false;
    const int N = s.N;
    for(size_t c = 0; c < (size_t)N * N; c++) heights[c] = INFINITY;
    /* the four vertices around the eye: +0 */
    const int i0 = (int)floorf(s.vci), j0 = (int)floorf(s.vcj);
    for(int dj = 0; dj < 2; dj++)
        for(int di = 0; di < 2; di++) vs_min(heights, N, i0 + di, j0 + dj, 0.f);
    #pragma omp parallel for num_threads(nthreads < 1 ? 1 : nthreads) schedule(dynamic, 64)
    for(int k = 0; k < 4 * N - 4; k++)
    {
        int ti, tj;
        vs_target(N, k, &ti, &tj);
        vs_ray_heights(&s, ti, tj, heights);
    }
    return true;
}
