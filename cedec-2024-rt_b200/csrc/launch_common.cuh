// launch_common.cuh — thread mapping, row slabs, shadow-ray queue plumbing and argument checks shared by the
// kernel translation units (kernels_dropin.cu: the reference's per-kernel entry points on AoS buffers;
// kernels_fast.cu: the fused frame on SoA buffers).
#pragma once
#include "ctx.cuh"
#include "shadow_queue.cuh"

namespace crt
{
constexpr int kTileW = 32, kTileH = 8;

// pixel of this thread
struct TilePix
{
    Pix px;
    bool in;
};
// rows [y0, y1) of the image are processed (multi-GPU row slabs: crt_set_row_range); pixel coordinates stay global
struct Rows
{
    int y0, y1;
};
__device__ __forceinline__ TilePix this_pixel(int W, int H, Rows rows)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int xi = blockIdx.x * kTileW + (warp & 3) * 8 + (lane & 7);
    const int yi = rows.y0 + blockIdx.y * kTileH + (warp >> 2) * 4 + (lane >> 3);
    return {make_pix(xi, yi, W, H), xi < W && yi < rows.y1};
}
static dim3 tile_grid(int W, Rows r)
{
    const int ny = (r.y1 - r.y0 + kTileH - 1) / kTileH;
    return dim3((W + kTileW - 1) / kTileW, ny > 0 ? ny : 1);  // an empty slab still launches one (idle) row of tiles
}
static Rows rows_of(const crt_ctx* ctx, int H)
{
    Rows r{ctx->row_begin, ctx->row_end < 0 || ctx->row_end > H ? H : ctx->row_end};
    if (r.y0 < 0) r.y0 = 0;
    if (r.y0 > r.y1) r.y0 = r.y1;
    return r;
}

__device__ __forceinline__ ShadowRay to_shadow_ray(const DeferredRay& d, int pix)
{
    ShadowRay r;
    r.ox = d.org.x; r.oy = d.org.y; r.oz = d.org.z;
    r.pix = (uint32_t)pix;
    r.dx = d.dir.x; r.dy = d.dir.y; r.dz = d.dir.z;
    r.ucw = 0.0f;
    r.bgx = r.bgy = r.bgz = r.pad0 = r.rx = r.ry = r.rz = r.pad1 = 0.0f;
    return r;
}
static __global__ void __launch_bounds__(256) k_build_light_table(uint32_t n, const float* tris60, const uint32_t* lights, LightRec* table)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) table[i] = make_light_rec(tris60, lights[i], n);
}
}  // namespace crt

namespace crt
{
inline size_t bsize(const crt_buffer& b) { return (size_t)CRT_BUFFER_SIZE(b); }
inline f3 to_f3(const crt_float3& v) { return f3{v.x, v.y, v.z}; }
inline unsigned sweep_blocks(crt_ctx* ctx, size_t n)
{
    const size_t want = (n + 255) / 256, cap = (size_t)ctx->sm_count * 8;
    return (unsigned)(want < cap ? (want ? want : 1) : cap);
}

// ---- wavefront plumbing
// which = 1: the second queue (resolve rays of a frame whose tail overlaps the next frame, crt_set_frame_overlap)
static int queue_prepare(crt_ctx* ctx, size_t n_pixels, ShadowQueue* q, int which = 0)
{
    if (!ctx->queue_counters)
    {
        CRT_CUDA(cudaMalloc((void**)&ctx->queue_counters, 8 * sizeof(unsigned)));  // count, next, three 64-bit totals
        CRT_CUDA(cudaMemsetAsync(ctx->queue_counters, 0, 8 * sizeof(unsigned), ctx->stream));
    }
    void*& rays = which ? ctx->queue2_rays : ctx->queue_rays;
    size_t& capacity = which ? ctx->queue2_capacity : ctx->queue_capacity;
    if (capacity < n_pixels)
    {
        if (rays) CRT_CUDA(cudaFree(rays));
        rays = nullptr;
        capacity = 0;
        CRT_CUDA(cudaMalloc(&rays, n_pixels * sizeof(ShadowRay)));
        capacity = n_pixels;
    }
    if (which && !ctx->queue2_counters) CRT_CUDA(cudaMalloc((void**)&ctx->queue2_counters, 2 * sizeof(unsigned)));
    unsigned* counters = which ? ctx->queue2_counters : ctx->queue_counters;
    CRT_CUDA(cudaMemsetAsync(counters, 0, 2 * sizeof(unsigned), ctx->stream));
    q->rays = (ShadowRay*)rays;
    q->count = counters;
    q->next = counters + 1;
    q->capacity = (uint32_t)capacity;
    q->total = (unsigned long long*)(ctx->queue_counters + 2);
    return CRT_OK;
}
template <int EPI>
static int queue_trace(crt_ctx* ctx, crt_geometry geom, const ShadowQueue& q, const ShadowSink& sink, cudaStream_t on = nullptr)
{
    static int blocks_per_sm = 0;
    if (!blocks_per_sm)
    {
        CRT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, k_trace_shadow_queue<EPI>, kShadowWarps * 32, 0));
        if (blocks_per_sm < 1) blocks_per_sm = 1;
        // tuning hook: fewer resident blocks per SM for the resolve tracer (which runs beside the next frame's head when
        // frames overlap) or for the others — leaves room for the kernels of the other streams
        if (const char* e = getenv(EPI == kEpiResolve ? "CRT_RESOLVE_BLOCKS_PER_SM" : "CRT_TRACE_BLOCKS_PER_SM"))
        {
            const int v = atoi(e);
            if (v >= 1 && v < blocks_per_sm) blocks_per_sm = v;
        }
    }
    cudaStream_t st = on ? on : ctx->stream;
    k_trace_shadow_queue<EPI><<<blocks_per_sm * ctx->sm_count, kShadowWarps * 32, 0, st>>>(geom->view(), q, sink);
    return check_launch(ctx, EPI == kEpiCountVisible ? "trace_ao" : EPI == kEpiBitmask ? "trace_shadow" : (EPI == kEpiReservoirVisibility || EPI == kEpiSoaVisibility) ? "trace_visibility_reuse" : "trace_resolve", st);
}
// power-proportional slot table of 2^log2_slots records (geometry.cu)
int build_light_slots(crt_ctx* ctx, crt_geometry geom, const float* tris60, const uint32_t* lights, uint32_t n, int log2_slots,
                      LightRec* table);
// light records for (geometry, light list, selection mode, K): one per light (uniform selection) or one per slot
// (CRT_LIGHTS_POWER); *n_out is the count LightsTable draws over, n or K.  Rebuilt when any of the four changes.
static int light_table_for(crt_ctx* ctx, crt_geometry geom, const float* tris60, const uint32_t* lights, size_t n,
                           const LightRec** out, uint32_t* n_out)
{
    const bool power = ctx->light_mode == CRT_LIGHTS_POWER && n > 0;
    const int k = power ? light_slots_log2(n, ctx->light_log2) : -1;
    CRT_REQUIRE(!power || k >= 0, n > ((size_t)1 << kMaxLightSlotsLog2) ? "power light selection takes at most 2^23 lights"
                                                                          : "log2_slots: 2^k must be at least the light count, k at most 23");
    const size_t count = power ? (size_t)1 << k : n;
    if (geom->light_table_key != lights || geom->light_table_n != n || geom->light_table_log2 != k)
    {
        geom->light_table_key = nullptr;
        if (geom->light_table_cap < (count ? count : 1))  // a rebuild of the same size (refit, new emission) reuses the memory
        {
            if (geom->light_table) CRT_CUDA(cudaFree(geom->light_table));
            geom->light_table = nullptr;
            geom->light_table_cap = 0;
            CRT_CUDA(cudaMalloc(&geom->light_table, (count ? count : 1) * sizeof(LightRec)));
            geom->light_table_cap = count ? count : 1;
        }
        if (power)
        {
            const int rc = build_light_slots(ctx, geom, tris60, lights, (uint32_t)n, k, (LightRec*)geom->light_table);
            if (rc != CRT_OK) return rc;
        }
        else if (n)
        {
            k_build_light_table<<<div_up(n, 256), 256, 0, ctx->stream>>>((uint32_t)n, tris60, lights, (LightRec*)geom->light_table);
            const int rc = check_launch(ctx, "build_light_table");
            if (rc != CRT_OK) return rc;
        }
        geom->light_table_key = lights;
        geom->light_table_n = n;
        geom->light_table_log2 = k;
        geom->light_table_gen++;
    }
    *out = (const LightRec*)geom->light_table;
    *n_out = (uint32_t)count;
    return CRT_OK;
}
// every kernel that samples lights reads the table in power mode and with light tiles; in uniform mode CRT_LIGHT_TABLE=0
// reads lights[] instead
inline bool use_light_table(const crt_ctx* ctx) { return ctx->light_table || ctx->light_mode == CRT_LIGHTS_POWER || ctx->tiles_log2_s || ctx->tiles_log2_t; }
// presampled light tiles (geometry.cu)
int build_light_tiles(crt_ctx* ctx, const LightRec* src, uint32_t K, int frame, int log2_t, int log2_s, LightRec* tiles);
// the context's light tiles of `frame` over the source table (src, K) of `geom` (light_table_for), rebuilt on the context's
// stream when any of (geometry, source table, frame, T, S) changed.  Every kernel that reads the tiles runs on that stream
// too (the frame tail and the primary-ray prefetch read none), so a rebuild is ordered after the last frame's reads.
static int light_tiles_for(crt_ctx* ctx, crt_geometry geom, const LightRec* src, uint32_t K, int frame, const LightRec** out)
{
    const int a = ctx->tiles_log2_t, b = ctx->tiles_log2_s;
    const unsigned long long key[5] = {geom->serial, geom->light_table_gen, (unsigned long long)(unsigned)frame,
                                       (unsigned long long)a, (unsigned long long)b};
    bool same = ctx->tiles_valid;
    for (int i = 0; i < 5; i++) same = same && ctx->tiles_key[i] == key[i];
    if (!same)
    {
        ctx->tiles_valid = false;
        const size_t count = (size_t)1 << (a + b);
        if (ctx->tiles_cap < count)
        {
            if (ctx->tiles) CRT_CUDA(cudaFree(ctx->tiles));
            ctx->tiles = nullptr;
            ctx->tiles_cap = 0;
            CRT_CUDA(cudaMalloc(&ctx->tiles, count * sizeof(LightRec)));
            ctx->tiles_cap = count;
        }
        const int rc = build_light_tiles(ctx, src, K, frame, a, b, (LightRec*)ctx->tiles);
        if (rc != CRT_OK) return rc;
        for (int i = 0; i < 5; i++) ctx->tiles_key[i] = key[i];
        ctx->tiles_valid = true;
    }
    *out = (const LightRec*)ctx->tiles;
    return CRT_OK;
}
inline bool light_tiles_on(const crt_ctx* ctx, uint32_t n_lights) { return (ctx->tiles_log2_t || ctx->tiles_log2_s) && n_lights; }
}  // namespace crt

namespace crt
{
// force the (lazily loaded) kernels of a translation unit into the context; see crt_slab_set_links
// slots != nullptr: examples 08 / 09 select lights from the power-proportional slot table (n_slots records)
int path_trace_wavefront(crt_ctx* ctx, int example, int W, int H, int frame, crt_geometry geom, const float* tris60,
                         const uint32_t* lights, uint32_t n_lights, const LightRec* slots, uint32_t n_slots, crt_raygen raygen,
                         crt_options options, crt_float4* accum, unsigned long long* counters);
int raycast_or_prefetched(crt_ctx* ctx, int W, int H, crt_geometry geom, crt_buffer triangles, crt_raygen raygen, crt_buffer visibility);
int raycast_rows(crt_ctx* ctx, int W, int H, crt_geometry geom, crt_raygen raygen, Rows rows, crt_visibility* vis, const char* what);
int tone_mapping_on(crt_ctx* ctx, cudaStream_t st, crt_buffer pixels, crt_buffer accumulation, int W, int H);
int preload_fused_kernels();
int preload_dropin_kernels();
}  // namespace crt

#define CRT_CHECK_IMAGE(W, H) CRT_REQUIRE((W) > 0 && (H) > 0 && (size_t)(W) * (size_t)(H) < 0x7fffffffull, "bad image size")
#define CRT_CHECK_BUF(b, n, what) CRT_REQUIRE((b).data != nullptr && bsize(b) >= (size_t)(n), what " buffer too small or null")

