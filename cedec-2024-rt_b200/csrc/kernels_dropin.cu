// kernels_dropin.cu — the reference's kernel entry points on the reference's own AoS buffers
// ("drop-in mode"): same parameter lists as the KERNELs of examples/10_restir_di/10_restir_di.cu,
// common/kernels/common.cu, 06_ao_hiprt.cu, 07_pt.cu, 08_nee.cu and 09_ris.cu, so the unmodified host
// loop (10_restir_di.cpp:229-380) can drive them through crt_launch / the crt_* exports.
//
// Thread mapping: one thread per pixel like the reference, but a 256-thread block covers a 32x8 pixel
// tile and each warp an 8x4 sub-tile (the reference's linear tid gives 32x1 strips): primary rays of a
// warp stay coherent and the Gaussian neighbourhoods of a block overlap in L1.  Randomness is keyed on
// (xi, yi, frame, stage), so the mapping does not change any result.
#include "launch_common.cuh"

namespace crt
{
__global__ void __launch_bounds__(256) k_raycast(int W, int H, Rows rows, Bvh bvh, crt_raygen raygen, crt_visibility* vis)
{
    const TilePix t = this_pixel(W, H, rows);
    if (t.in) px_raycast(t.px, W, H, bvh, raygen, vis);
}
// the same rays, each walk seeded with the triangle the pixel's record names before the call (restir_pixel.cuh:
// px_raycast_hinted); launched when the host hands in the triangle array the tree was built over
__global__ void __launch_bounds__(256) k_raycast_hinted(int W, int H, Rows rows, Bvh bvh, crt_raygen raygen, crt_visibility* vis,
                                                        const float* tris60, uint32_t n_tris)
{
    const TilePix t = this_pixel(W, H, rows);
    // a seeded walk accepts (almost) no triangle any more, and triangle postponing — which waits for more lanes before it
    // runs the test — only delays it: 1.695 -> 1.672 ms without (profiles/r2/tuning.txt, batch 33)
    bvh.postpone_ratio = 0.0f;
    if (t.in) px_raycast_hinted(t.px, W, H, bvh, raygen, vis, tris60, n_tris);
}
// WF: emit the visibility-reuse ray into the queue instead of walking it here (shadow_queue.cuh)
// SH: use_shadowed_target_function may be set (traversal code inside the target function); the common SH = false
// instantiation has none, which takes the walk's stack and ~40 registers out of the reservoir kernels
template <bool SH>
__device__ __forceinline__ Opt kernel_opt(const crt_options& options)
{
    Opt o = make_opt(options);
    if (!SH) o.shadowed = false;
    return o;
}
template <class L, bool WF, bool SH>
__global__ void __launch_bounds__(256)
    k_generate_candidate(int W, int H, Rows rows, int frame, Bvh bvh, const float* tris60, const crt_visibility* vis, f3 eye,
                         L lights, crt_options options, crt_reservoir* out, ShadowQueue q)
{
    const TilePix t = this_pixel(W, H, rows);
    DeferredRay d{false, {0, 0, 0}, {0, 0, 0}};
    if (t.in) d = px_generate_candidate(t.px, frame, bvh, tris60, vis, eye, lights, kernel_opt<SH>(options), AosStore{out}, WF);
    if (WF) queue_push(q, d.want, to_shadow_ray(d, t.px.idx), d.decided);
}
// RW: the reuse weights (crt_set_reuse_weights), CRT_REUSE_REFERENCE or CRT_REUSE_UNBIASED
template <int MODE, bool SH, int RW>
__global__ void __launch_bounds__(256)
    k_temporal(int W, int H, Rows rows, int frame, Bvh bvh, const float* tris60, const crt_visibility* vis, f3 eye,
               crt_options options, const crt_reservoir* prev, crt_reservoir* cur)
{
    const TilePix t = this_pixel(W, H, rows);
    if (t.in)
        px_temporal<Math<MODE>, RW>(t.px, frame, bvh, tris60, vis, eye, kernel_opt<SH>(options),
                                    AosStore{const_cast<crt_reservoir*>(prev)}, AosStore{cur});
}
// the same with reprojection into the previous frame's camera (extension; reads `prev` anywhere in the image).  RW =
// CRT_REUSE_UNBIASED reads the previous frame's Visibility `prev_vis` at the history pixel; the reference's merge ignores it
// (the last parameter, so that the reference instantiations keep their code)
template <int MODE, bool SH, int RW>
__global__ void __launch_bounds__(256)
    k_temporal_reprojected(int W, int H, Rows rows, int frame, Bvh bvh, const float* tris60, const crt_visibility* vis, f3 eye,
                           crt_options options, crt_raygen prev_cam, const crt_reservoir* prev, crt_reservoir* cur,
                           const crt_visibility* prev_vis)
{
    const TilePix t = this_pixel(W, H, rows);
    if (t.in)
        px_temporal<Math<MODE>, RW>(t.px, frame, bvh, tris60, vis, eye, kernel_opt<SH>(options),
                                    AosStore{const_cast<crt_reservoir*>(prev)}, AosStore{cur}, &prev_cam, W, H, prev_vis);
}
// 10_restir_di.cu:239-254 (the first buffer is the source).  Every pixel is copied, so the bottom-up
// index permutation does not matter: plain word copy.
__global__ void __launch_bounds__(256) k_save_temporal(size_t n_words, const uint32_t* src, uint32_t* dst)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}
template <int MODE, bool SH, int RW>
__global__ void __launch_bounds__(256)
    k_spatial(int W, int H, Rows rows, int frame, int pass, Bvh bvh, const float* tris60, const crt_visibility* vis, f3 eye,
              crt_options options, const crt_reservoir* in, crt_reservoir* out)
{
    const TilePix t = this_pixel(W, H, rows);
    if (t.in)
        px_spatial<Math<MODE>, RW>(t.px, W, H, frame, pass, bvh, tris60, vis, eye, kernel_opt<SH>(options),
                                   AosStore{const_cast<crt_reservoir*>(in)}, AosStore{out});
}
template <bool WF>
__global__ void __launch_bounds__(256)
    k_resolve(crt_float4* accum, int W, int H, Rows rows, Bvh bvh, const float* tris60, const crt_visibility* vis, f3 eye,
              crt_options options, const crt_reservoir* res, ShadowQueue q)
{
    const TilePix t = this_pixel(W, H, rows);
    DeferredRay d{false, {0, 0, 0}, {0, 0, 0}};
    DeferredShade sh{{0, 0, 0}, {0, 0, 0}, 0.0f};
    if (t.in)
        d = px_resolve(t.px, accum, bvh, tris60, vis, eye, make_opt(options), AosStore{const_cast<crt_reservoir*>(res)},
                       WF ? &sh : nullptr);
    if (WF)
    {
        ShadowRay r = to_shadow_ray(d, t.px.idx);
        r.ucw = sh.ucw;
        r.bgx = sh.bg.x; r.bgy = sh.bg.y; r.bgz = sh.bg.z;
        r.rx = sh.rad.x; r.ry = sh.rad.y; r.rz = sh.rad.z;
        queue_push(q, d.want, r);
    }
}

// ---- common/kernels/common.cu:4-17 and :30-74 (every pixel is touched: plain linear sweeps)
__global__ void __launch_bounds__(256) k_clear(size_t n, float4* buf)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        buf[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}
template <int MODE>
__global__ void __launch_bounds__(256) k_tone_mapping(size_t n, uint32_t* pixels, const float4* accum)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    {
        const float4 a = accum[i];
        pixels[i] = tone_map_rgba8<Math<MODE>>(f4{a.x, a.y, a.z, a.w});
    }
}
// rays traced inside the single-kernel examples (crt_inline_rays_traced): one atomic per warp
__device__ __forceinline__ void count_rays(unsigned long long* counters, uint32_t n_closest, uint32_t n_shadow)
{
    const uint32_t c = __reduce_add_sync(0xffffffffu, n_closest), s = __reduce_add_sync(0xffffffffu, n_shadow);
    if ((threadIdx.x & 31) == 0)
    {
        if (c) atomicAdd(counters + 0, (unsigned long long)c);
        if (s) atomicAdd(counters + 1, (unsigned long long)s);
    }
}
template <int EX, int MODE, class LS>
__global__ void __launch_bounds__(256)
    k_path_trace(int W, int H, Rows rows, int frame, Bvh bvh, const float* tris60, const typename LS::Elem* lights, uint32_t n_lights,
                 crt_raygen raygen, crt_options options, crt_float4* accum, unsigned long long* ray_counters)
{
    const TilePix t = this_pixel(W, H, rows);
    uint32_t n = 0;
    if (t.in)
        n = px_path_trace<EX, Math<MODE>, LS>(t.px, W, H, frame, bvh, tris60, lights, n_lights, raygen, make_opt(options), accum);
    count_rays(ray_counters, n & 0xffffu, n >> 16);
}
template <int MODE>
__global__ void __launch_bounds__(256, 3)  // 80 registers: the walk-step loop would otherwise take 128 and halve the resident warps
    k_ao(uint32_t* pixels, crt_raygen raygen, int W, int H, Rows rows, Bvh bvh, const float* tris60, int n_rays,
         unsigned long long* ray_counters)
{
    const TilePix t = this_pixel(W, H, rows);
    uint32_t ao_rays = 0;
    if (t.in) pixels[t.px.idx] = px_ao<Math<MODE>>(t.px, raygen, W, H, bvh, tris60, n_rays, ao_rays);
    count_rays(ray_counters, t.in ? 1u : 0u, ao_rays);
}
// ---- 06_ao_hiprt.cu:35-91 as a wavefront (the shape the fused frame gives its shadow rays): the per-pixel kernel traces
// the primary ray and only *emits* the n_rays hemisphere rays — compact 32-byte records, one queue reservation per warp,
// ray i of the warp's hit pixels next to each other — the persistent kernel of shadow_queue.cuh walks them (t in
// [0, FLT_MAX], near children first) and counts the unoccluded ones per pixel, and a third kernel turns the counts into
// pixels.  Same rays, same random numbers, same counts as the single kernel (px_ao), which stays for CRT_WAVEFRONT=0.
constexpr uint32_t kAoSky = 0xffffffffu;  // visible_count of a pixel whose primary ray missed
template <int MODE>
__global__ void __launch_bounds__(256)
    k_ao_emit(crt_raygen raygen, int W, int H, Rows rows, Bvh bvh, const float* tris60, int n_rays, ShadowQueue q,
              uint32_t* visible_count, unsigned long long* ray_counters)
{
    const TilePix t = this_pixel(W, H, rows);
    const Pix px = t.px;
    bool hit = false;
    f3 n{0, 0, 0}, t0{0, 0, 0}, t1{0, 0, 0}, ao_ro{0, 0, 0};
    Pcg rng(0, hash_pcg3(px.xi, px.yi, 42));
    if (t.in)
    {
        f3 ro, rd;
        primary_ray(raygen, px, W, H, ro, rd);
        Hit h;
        hit = trace<false>(bvh, ro, rd, 0.0f, kFltMax, h);
        if (hit)
        {
            const TriRef tri = tri_at(tris60, h.prim);
            const f3 v0 = tri.v(0), v1 = tri.v(1), v2 = tri.v(2);
            n = tri_normal(v0, v1, v2);
            if (0.0f < dot(n, rd)) n = -n;
            t0 = normalize(v1 - v0);
            t1 = cross(t0, n);
            ao_ro = ro + rd * h.t + n * 0.0001f;
        }
        visible_count[px.idx] = hit ? 0u : kAoSky;
    }
    const unsigned mask = __ballot_sync(0xffffffffu, hit);
    count_rays(ray_counters, t.in ? 1u : 0u, hit ? (uint32_t)n_rays : 0u);
    if (mask == 0) return;
    const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
    const uint32_t n_hit = (uint32_t)__popc(mask), rank = (uint32_t)__popc(mask & ((1u << lane) - 1u));
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(q.count, n_hit * (uint32_t)n_rays);
    base = __shfl_sync(0xffffffffu, base, leader);
    if (!hit) return;
    float4* out = (float4*)q.rays;
    for (int i = 0; i < n_rays; i++)
    {
        const float r0 = rng.next_f();
        const float r1 = rng.next_f();
        const float r2 = rng.next_f();
        const f3 s = sample_hemisphere<Math<MODE>>(r0, r1, r2);
        const f3 ao_rd = t0 * s.x + t1 * s.z + n * s.y;
        float4* dst = out + ((size_t)base + (size_t)i * n_hit + rank) * 2;
        dst[0] = make_float4(ao_ro.x, ao_ro.y, ao_ro.z, __uint_as_float((uint32_t)px.idx));
        dst[1] = make_float4(ao_rd.x, ao_rd.y, ao_rd.z, 0.0f);
    }
}
template <int MODE>
__global__ void __launch_bounds__(256) k_ao_finish(size_t first, size_t n, uint32_t* pixels, const uint32_t* visible_count, int n_rays)
{
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (size_t)gridDim.x * blockDim.x)
    {
        const size_t i = first + k;
        const uint32_t cnt = visible_count[i];
        uint32_t c = 32u;  // background (06_ao_hiprt.cu:57-60)
        if (cnt != kAoSky)
        {
            const float ao = (float)(int)cnt / (float)n_rays;
            c = (uint32_t)(Math<MODE>::pow(ao, 1.0f / 2.2f) * 255.0f) & 0xffu;
        }
        pixels[i] = c | (c << 8) | (c << 16) | (255u << 24);
    }
}

// the kernels of this file the fused frame launches (crt_slab_set_links loads them ahead of any spinning wait)
int preload_dropin_kernels()
{
    cudaFuncAttributes a;
    CRT_CUDA(cudaFuncGetAttributes(&a, k_raycast));
    CRT_CUDA(cudaFuncGetAttributes(&a, k_raycast_hinted));
    CRT_CUDA(cudaFuncGetAttributes(&a, k_tone_mapping<0>));
    CRT_CUDA(cudaFuncGetAttributes(&a, k_tone_mapping<1>));
    CRT_CUDA(cudaFuncGetAttributes(&a, k_clear));
    return CRT_OK;
}
}  // namespace crt

// ======================================================================================= C ABI
using namespace crt;

extern "C" int crt_raycast(crt_ctx* ctx, int W, int H, crt_geometry geom, crt_buffer triangles, crt_raygen raygen,
                           crt_buffer visibility_buffer)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(visibility_buffer, (size_t)W * H, "visibility");
    // The reference's raycast does not read `triangles` (10_restir_di.cu:9-34).  Here it is the licence for the hinted walk:
    // when it is the very array the tree was built over, the record each pixel already holds seeds its walk.
    if (triangles.data == nullptr || triangles.data != (const void*)geom->src) ctx->hint_tris = nullptr;
    if (ctx->raycast_hint && triangles.data != nullptr && triangles.data == (const void*)geom->src && geom->n_tris)
        ctx->hint_tris = geom->src;
    return raycast_rows(ctx, W, H, geom, raygen, rows_of(ctx, H), (crt_visibility*)visibility_buffer.data, "raycast");
}

// ---- primary rays of the next frame, ahead of time (frame overlap; include/cedecrt.h)
extern "C" int crt_restir_prefetch_raycast(crt_ctx* ctx, int W, int H, crt_geometry geom, crt_raygen raygen)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    CRT_CHECK_IMAGE(W, H);
    if (!ctx->overlap || ctx->profiling) return CRT_OK;  // strictly serial frames: the next crt_restir_frame_begin traces its own rays
    const size_t n = (size_t)W * H;
    if (!ctx->head_stream)
    {
        CRT_CUDA(cudaSetDevice(ctx->device));
        CRT_CUDA(cudaStreamCreateWithFlags(&ctx->head_stream, cudaStreamNonBlocking));
        CRT_CUDA(cudaEventCreateWithFlags(&ctx->ev_ray_ready, cudaEventDisableTiming));
        CRT_CUDA(cudaEventCreateWithFlags(&ctx->ev_vis_consumed, cudaEventDisableTiming));
    }
    if (ctx->vis_next_pixels < n) CRT_CUDA(cudaStreamSynchronize(ctx->head_stream));  // the last prefetch may still write the buffer
    bool fresh = false;
    int rc = grow(ctx->vis_next, ctx->vis_next_pixels, n, n * sizeof(crt_visibility), &fresh);
    if (rc != CRT_OK) return rc;
    if (fresh) CRT_CUDA(cudaMemsetAsync(ctx->vis_next, 0xff, n * sizeof(crt_visibility), ctx->head_stream));  // index -1: no hint yet
    if (ctx->vis_consumed_pending)  // the frame in flight may still be copying the previous prefetch out of the buffer
    {
        CRT_CUDA(cudaStreamWaitEvent(ctx->head_stream, ctx->ev_vis_consumed, 0));
        ctx->vis_consumed_pending = false;
    }
    const Rows rows = rows_of(ctx, H);
    // hinted when a frame of this context has shown the tree's own triangle array to be alive (crt_raycast above); the
    // buffer is the context's own and holds the previous prefetch, or index -1 everywhere after its allocation
    rc = raycast_rows(ctx, W, H, geom, raygen, rows, (crt_visibility*)ctx->vis_next, "raycast", ctx->head_stream);
    if (rc != CRT_OK) return rc;
    CRT_CUDA(cudaEventRecord(ctx->ev_ray_ready, ctx->head_stream));
    ctx->ray_next_cam = raygen;
    ctx->ray_next_geom = geom->serial;
    ctx->ray_next_dims[0] = W; ctx->ray_next_dims[1] = H; ctx->ray_next_dims[2] = rows.y0; ctx->ray_next_dims[3] = rows.y1;
    ctx->ray_next_valid = true;
    return CRT_OK;
}
namespace crt
{
// crt_raycast, or — when the very same rays were traced ahead of time — a copy of their Visibility rows
int raycast_or_prefetched(crt_ctx* ctx, int W, int H, crt_geometry geom, crt_buffer triangles, crt_raygen raygen, crt_buffer visibility)
{
    const Rows rows = rows_of(ctx, H);
    // every frame renews (or withdraws) the licence for the prefetch's hints: the host has just handed in its triangle array
    ctx->hint_tris = (triangles.data != nullptr && triangles.data == (const void*)geom->src) ? (const void*)geom->src : nullptr;
    const bool hit = ctx->ray_next_valid && ctx->ray_next_geom == geom->serial && !memcmp(&ctx->ray_next_cam, &raygen, sizeof raygen) &&
                     ctx->ray_next_dims[0] == W && ctx->ray_next_dims[1] == H && ctx->ray_next_dims[2] == rows.y0 &&
                     ctx->ray_next_dims[3] == rows.y1 && !ctx->profiling;
    ctx->ray_next_valid = false;
    if (!hit) return crt_raycast(ctx, W, H, geom, triangles, raygen, visibility);
    CRT_CHECK_BUF(visibility, (size_t)W * H, "visibility");
    const size_t first = (size_t)(H - rows.y1) * W, count = (size_t)(rows.y1 - rows.y0) * W;
    CRT_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_ray_ready, 0));
    if (count)
        CRT_CUDA(cudaMemcpyAsync((crt_visibility*)visibility.data + first, (const crt_visibility*)ctx->vis_next + first,
                                 count * sizeof(crt_visibility), cudaMemcpyDeviceToDevice, ctx->stream));
    CRT_CUDA(cudaEventRecord(ctx->ev_vis_consumed, ctx->stream));
    ctx->vis_consumed_pending = true;
    return CRT_OK;
}
// primary rays of rows [rows.y0, rows.y1) into `vis` on stream `on` (default: the context's), each walk seeded with the
// pixel's record (k_raycast_hinted) while the context holds the licence for the tree's own triangle array (ctx->hint_tris,
// set or cleared by crt_raycast and raycast_or_prefetched)
int raycast_rows(crt_ctx* ctx, int W, int H, crt_geometry geom, crt_raygen raygen, Rows rows, crt_visibility* vis, const char* what,
                 cudaStream_t on)
{
    cudaStream_t st = on ? on : ctx->stream;
    if (ctx->raycast_hint && ctx->hint_tris != nullptr && ctx->hint_tris == (const void*)geom->src && geom->n_tris)
        k_raycast_hinted<<<tile_grid(W, rows), 256, 0, st>>>(W, H, rows, geom->view(), raygen, vis, (const float*)geom->src,
                                                             (uint32_t)geom->n_tris);
    else
        k_raycast<<<tile_grid(W, rows), 256, 0, st>>>(W, H, rows, geom->view(), raygen, vis);
    return check_launch(ctx, what, on);
}
}  // namespace crt

extern "C" int crt_generate_candidate(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom, crt_buffer triangles,
                                      crt_buffer visibility_buffer, crt_float3 eye, crt_buffer lights,
                                      crt_options options, crt_buffer reservoirs)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(visibility_buffer, (size_t)W * H, "visibility");
    CRT_CHECK_BUF(reservoirs, (size_t)W * H, "reservoir");
    CRT_REQUIRE(triangles.data != nullptr, "null triangle buffer");
    CRT_REQUIRE(bsize(lights) == 0 || lights.data != nullptr, "null light buffer");
    CRT_REQUIRE(bsize(lights) < 0xffffffffull, "too many lights");
    const Rows rows = rows_of(ctx, H);
    const float* tris60 = (const float*)triangles.data;
    const crt_visibility* vis = (const crt_visibility*)visibility_buffer.data;
    crt_reservoir* res = (crt_reservoir*)reservoirs.data;
    const uint32_t n_lights = (uint32_t)bsize(lights);
    const bool wf = ctx->wavefront && options.use_visibility_reuse;
    ShadowQueue q{nullptr, nullptr, nullptr, 0};
    if (wf)
    {
        const int rc = queue_prepare(ctx, (size_t)(rows.y1 - rows.y0) * W, &q);
        if (rc != CRT_OK) return rc;
    }
    const dim3 grid = tile_grid(W, rows);
    auto launch = [&](auto L)
    {
        with_flag(wf, [&](auto WF)
        {
            with_flag(options.use_shadowed_target_function != 0, [&](auto SH)
            {
                k_generate_candidate<decltype(L), WF, SH><<<grid, 256, 0, ctx->stream>>>(W, H, rows, frame, geom->view(), tris60, vis,
                                                                                          to_f3(eye), L, options, res, q);
            });
        });
    };
    if (use_light_table(ctx))
    {
        const LightRec* table = nullptr;
        uint32_t n_slots = 0;
        int rc = light_table_for(ctx, geom, tris60, (const uint32_t*)lights.data, n_lights, &table, &n_slots);
        if (rc != CRT_OK) return rc;
        if (light_tiles_on(ctx, n_lights))  // crt_set_light_tiles: the candidates draw from the pixel's tile of this frame
        {
            const LightRec* tiles = nullptr;
            rc = light_tiles_for(ctx, geom, table, n_slots, frame, &tiles);
            if (rc != CRT_OK) return rc;
            launch(LightsTiles{tiles, (uint32_t)ctx->tiles_log2_t, (uint32_t)ctx->tiles_log2_s});
        }
        else launch(LightsTable{table, n_slots});
    }
    else launch(LightsIndexed{tris60, (const uint32_t*)lights.data, n_lights});
    int rc = check_launch(ctx, "generate_candidate");
    if (rc != CRT_OK || !wf) return rc;
    return queue_trace<kEpiReservoirVisibility>(ctx, geom, q, ShadowSink{res, nullptr, 0, nullptr});
}

extern "C" int crt_light_sampling_table(crt_ctx* ctx, crt_geometry geom, crt_buffer lights, const void** d_records, uint32_t* n_slots)
{
    CRT_REQUIRE(ctx && geom && d_records && n_slots, "null argument");
    CRT_REQUIRE(bsize(lights) == 0 || lights.data != nullptr, "null light buffer");
    CRT_REQUIRE(bsize(lights) < 0xffffffffull, "too many lights");
    CRT_REQUIRE(geom->src != nullptr, "geometry has no triangle array");
    CRT_JOIN_TAIL(ctx);
    const LightRec* table = nullptr;
    const int rc = light_table_for(ctx, geom, (const float*)geom->src, (const uint32_t*)lights.data, bsize(lights), &table, n_slots);
    if (rc != CRT_OK) return rc;
    *d_records = table;
    return CRT_OK;
}

extern "C" int crt_light_tiles(crt_ctx* ctx, crt_geometry geom, crt_buffer lights, int frame, const void** d_records,
                               uint32_t* n_tiles, uint32_t* tile_size)
{
    CRT_REQUIRE(ctx && geom && d_records && n_tiles && tile_size, "null argument");
    CRT_REQUIRE(bsize(lights) > 0 && lights.data != nullptr, "light tiles need a non-empty light buffer");
    CRT_REQUIRE(bsize(lights) < 0xffffffffull, "too many lights");
    CRT_REQUIRE(geom->src != nullptr, "geometry has no triangle array");
    CRT_REQUIRE(light_tiles_on(ctx, 1), "light tiles are off (crt_set_light_tiles)");
    CRT_JOIN_TAIL(ctx);
    const LightRec* table = nullptr;
    uint32_t K = 0;
    int rc = light_table_for(ctx, geom, (const float*)geom->src, (const uint32_t*)lights.data, bsize(lights), &table, &K);
    if (rc != CRT_OK) return rc;
    const LightRec* tiles = nullptr;
    rc = light_tiles_for(ctx, geom, table, K, frame, &tiles);
    if (rc != CRT_OK) return rc;
    *d_records = tiles;
    *n_tiles = 1u << ctx->tiles_log2_t;
    *tile_size = 1u << ctx->tiles_log2_s;
    return CRT_OK;
}

// the temporal merge of the three entry points below: in place (prev_cam null) or reprojected into the previous camera,
// where prev_vis is the previous frame's Visibility (null: not given; CRT_REUSE_UNBIASED reads it at the history pixel)
static int temporal_resampling(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom, crt_buffer triangles,
                               crt_buffer visibility_buffer, crt_float3 eye, crt_options options, const crt_raygen* prev_cam,
                               const crt_visibility* prev_vis, crt_buffer previous_reservoirs, crt_buffer reservoirs, const char* what)
{
    const Rows rows = rows_of(ctx, H);
    const float* tris60 = (const float*)triangles.data;
    const crt_visibility* vis = (const crt_visibility*)visibility_buffer.data;
    const crt_reservoir* prev = (const crt_reservoir*)previous_reservoirs.data;
    crt_reservoir* cur = (crt_reservoir*)reservoirs.data;
    with_math_reuse(ctx->math_mode == CRT_MATH_EXACT, ctx->reuse_mode, [&](auto MODE, auto RW)
    {
        with_flag(options.use_shadowed_target_function != 0, [&](auto SH)
        {
            if (prev_cam)
                k_temporal_reprojected<MODE, SH, RW><<<tile_grid(W, rows), 256, 0, ctx->stream>>>(
                    W, H, rows, frame, geom->view(), tris60, vis, to_f3(eye), options, *prev_cam, prev, cur, prev_vis);
            else
                k_temporal<MODE, SH, RW><<<tile_grid(W, rows), 256, 0, ctx->stream>>>(W, H, rows, frame, geom->view(), tris60, vis,
                                                                                   to_f3(eye), options, prev, cur);
        });
    });
    return check_launch(ctx, what);
}

extern "C" int crt_temporal_resampling(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom, crt_buffer triangles,
                                       crt_buffer visibility_buffer, crt_float3 eye, crt_options options,
                                       crt_buffer previous_reservoirs, crt_buffer reservoirs)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(visibility_buffer, (size_t)W * H, "visibility");
    CRT_CHECK_BUF(previous_reservoirs, (size_t)W * H, "previous reservoir");
    CRT_CHECK_BUF(reservoirs, (size_t)W * H, "reservoir");
    CRT_REQUIRE(triangles.data != nullptr, "null triangle buffer");
    return temporal_resampling(ctx, W, H, frame, geom, triangles, visibility_buffer, eye, options, nullptr, nullptr,
                               previous_reservoirs, reservoirs, "temporal_resampling");
}

extern "C" int crt_temporal_resampling_reprojected(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom, crt_buffer triangles,
                                                   crt_buffer visibility_buffer, crt_float3 eye, crt_options options,
                                                   crt_raygen previous_raygen, crt_buffer previous_reservoirs,
                                                   crt_buffer reservoirs)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(visibility_buffer, (size_t)W * H, "visibility");
    CRT_CHECK_BUF(previous_reservoirs, (size_t)W * H, "previous reservoir");
    CRT_CHECK_BUF(reservoirs, (size_t)W * H, "reservoir");
    CRT_REQUIRE(previous_reservoirs.data != reservoirs.data, "reprojection reads other pixels of the previous buffer: it cannot run in place");
    CRT_REQUIRE(triangles.data != nullptr, "null triangle buffer");
    CRT_REQUIRE(ctx->reuse_mode != CRT_REUSE_UNBIASED, "unbiased reuse weights do not take a previous camera here: this call does not receive "
                                                       "the previous frame's surfaces (crt_temporal_resampling_reprojected_surfaces does)");
    return temporal_resampling(ctx, W, H, frame, geom, triangles, visibility_buffer, eye, options, &previous_raygen, nullptr,
                               previous_reservoirs, reservoirs, "temporal_resampling_reprojected");
}

extern "C" int crt_temporal_resampling_reprojected_surfaces(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom,
                                                            crt_buffer triangles, crt_buffer visibility_buffer, crt_float3 eye,
                                                            crt_options options, crt_raygen previous_raygen,
                                                            crt_buffer previous_visibility_buffer,
                                                            crt_buffer previous_reservoirs, crt_buffer reservoirs)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(visibility_buffer, (size_t)W * H, "visibility");
    CRT_CHECK_BUF(previous_visibility_buffer, (size_t)W * H, "previous visibility");
    CRT_CHECK_BUF(previous_reservoirs, (size_t)W * H, "previous reservoir");
    CRT_CHECK_BUF(reservoirs, (size_t)W * H, "reservoir");
    CRT_REQUIRE(previous_visibility_buffer.data != visibility_buffer.data,
                "the previous frame's Visibility must be a buffer of its own: this frame's raycast has overwritten it");
    CRT_REQUIRE(previous_reservoirs.data != reservoirs.data, "reprojection reads other pixels of the previous buffer: it cannot run in place");
    CRT_REQUIRE(triangles.data != nullptr, "null triangle buffer");
    return temporal_resampling(ctx, W, H, frame, geom, triangles, visibility_buffer, eye, options, &previous_raygen,
                               (const crt_visibility*)previous_visibility_buffer.data, previous_reservoirs, reservoirs,
                               "temporal_resampling_reprojected_surfaces");
}

extern "C" int crt_save_temporal_reservoir(crt_ctx* ctx, int W, int H, crt_buffer src, crt_buffer dst)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(src, (size_t)W * H, "source reservoir");
    CRT_CHECK_BUF(dst, (size_t)W * H, "destination reservoir");
    // rows [y0,y1) are the contiguous pixel range [(H-y1)*W, (H-y0)*W) of the bottom-up buffers
    const Rows r = rows_of(ctx, H);
    const size_t wpp = sizeof(crt_reservoir) / 4, first = (size_t)(H - r.y1) * W * wpp;
    const size_t n_words = (size_t)(r.y1 - r.y0) * W * wpp;
    if (n_words == 0) return CRT_OK;
    k_save_temporal<<<sweep_blocks(ctx, n_words), 256, 0, ctx->stream>>>(n_words, (const uint32_t*)src.data + first,
                                                                        (uint32_t*)dst.data + first);
    return check_launch(ctx, "save_temporal_reservoir");
}

extern "C" int crt_spatial_resampling(crt_ctx* ctx, int W, int H, int frame, int pass, crt_geometry geom,
                                      crt_buffer triangles, crt_buffer visibility_buffer, crt_float3 eye,
                                      crt_options options, crt_buffer previous_reservoirs, crt_buffer reservoirs)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(visibility_buffer, (size_t)W * H, "visibility");
    CRT_CHECK_BUF(previous_reservoirs, (size_t)W * H, "input reservoir");
    CRT_CHECK_BUF(reservoirs, (size_t)W * H, "output reservoir");
    CRT_REQUIRE(previous_reservoirs.data != reservoirs.data, "spatial_resampling cannot run in place");
    CRT_REQUIRE(triangles.data != nullptr, "null triangle buffer");
    const Rows rows = rows_of(ctx, H);
    with_math_reuse(ctx->math_mode == CRT_MATH_EXACT, ctx->reuse_mode, [&](auto MODE, auto RW)
    {
        with_flag(options.use_shadowed_target_function != 0, [&](auto SH)
        {
            k_spatial<MODE, SH, RW><<<tile_grid(W, rows), 256, 0, ctx->stream>>>(
                W, H, rows, frame, pass, geom->view(), (const float*)triangles.data, (const crt_visibility*)visibility_buffer.data,
                to_f3(eye), options, (const crt_reservoir*)previous_reservoirs.data, (crt_reservoir*)reservoirs.data);
        });
    });
    return check_launch(ctx, "spatial_resampling");
}

extern "C" int crt_resolve(crt_ctx* ctx, crt_buffer accumulation, int W, int H, crt_geometry geom,
                           crt_buffer triangles, crt_buffer visibility_buffer, crt_float3 eye, crt_options options,
                           crt_buffer reservoirs)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(accumulation, (size_t)W * H, "accumulation");
    CRT_CHECK_BUF(visibility_buffer, (size_t)W * H, "visibility");
    CRT_CHECK_BUF(reservoirs, (size_t)W * H, "reservoir");
    CRT_REQUIRE(triangles.data != nullptr, "null triangle buffer");
    CRT_JOIN_TAIL(ctx);
    const Rows rows = rows_of(ctx, H);
    crt_float4* accum = (crt_float4*)accumulation.data;
    ShadowQueue q{nullptr, nullptr, nullptr, 0};
    if (ctx->wavefront)
    {
        int rc = queue_prepare(ctx, (size_t)(rows.y1 - rows.y0) * W, &q);
        if (rc != CRT_OK) return rc;
        k_resolve<true><<<tile_grid(W, rows), 256, 0, ctx->stream>>>(accum, W, H, rows, geom->view(), (const float*)triangles.data,
                                                                    (const crt_visibility*)visibility_buffer.data, to_f3(eye),
                                                                    options, (const crt_reservoir*)reservoirs.data, q);
        rc = check_launch(ctx, "resolve");
        if (rc != CRT_OK) return rc;
        return queue_trace<kEpiResolve>(ctx, geom, q, ShadowSink{nullptr, accum, options.accumulate, nullptr});
    }
    k_resolve<false><<<tile_grid(W, rows), 256, 0, ctx->stream>>>(accum, W, H, rows, geom->view(), (const float*)triangles.data,
                                                                 (const crt_visibility*)visibility_buffer.data, to_f3(eye),
                                                                 options, (const crt_reservoir*)reservoirs.data, q);
    return check_launch(ctx, "resolve");
}

extern "C" int crt_clear(crt_ctx* ctx, crt_buffer buffer, int W, int H)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(buffer, (size_t)W * H, "accumulation");
    CRT_JOIN_TAIL(ctx);
    const Rows r = rows_of(ctx, H);
    const size_t n = (size_t)(r.y1 - r.y0) * W, first = (size_t)(H - r.y1) * W;
    if (n == 0) return CRT_OK;
    k_clear<<<sweep_blocks(ctx, n), 256, 0, ctx->stream>>>(n, (float4*)buffer.data + first);
    return check_launch(ctx, "clear");
}

namespace crt
{
int tone_mapping_on(crt_ctx* ctx, cudaStream_t st, crt_buffer pixels, crt_buffer accumulation, int W, int H)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(pixels, (size_t)W * H * 4, "pixel");
    CRT_CHECK_BUF(accumulation, (size_t)W * H, "accumulation");
    const Rows r = rows_of(ctx, H);
    const size_t n = (size_t)(r.y1 - r.y0) * W, first = (size_t)(H - r.y1) * W;
    if (n == 0) return CRT_OK;
    auto k = ctx->math_mode == CRT_MATH_EXACT ? k_tone_mapping<1> : k_tone_mapping<0>;
    k<<<sweep_blocks(ctx, n), 256, 0, st>>>(n, (uint32_t*)pixels.data + first, (const float4*)accumulation.data + first);
    return check_launch(ctx, "tone_mapping", st);
}
}  // namespace crt

extern "C" int crt_tone_mapping(crt_ctx* ctx, crt_buffer pixels, crt_buffer accumulation, int W, int H)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_JOIN_TAIL(ctx);
    return tone_mapping_on(ctx, ctx->stream, pixels, accumulation, W, H);
}

// two 64-bit device counters per context: closest-hit and shadow / AO rays traced by the single-kernel examples
static int inline_ray_counters(crt_ctx* ctx, unsigned long long** out)
{
    if (!ctx->inline_rays)
    {
        CRT_CUDA(cudaMalloc((void**)&ctx->inline_rays, 3 * sizeof(unsigned long long)));  // [2]: settled by the own-triangle pre-test
        CRT_CUDA(cudaMemsetAsync(ctx->inline_rays, 0, 3 * sizeof(unsigned long long), ctx->stream));
    }
    *out = ctx->inline_rays;
    return CRT_OK;
}
extern "C" int crt_inline_rays_traced(crt_ctx* ctx, unsigned long long out[2])
{
    CRT_REQUIRE(ctx && out, "null argument");
    out[0] = out[1] = 0;
    if (!ctx->inline_rays) return CRT_OK;
    CRT_CUDA(cudaMemcpyAsync(out, ctx->inline_rays, 2 * sizeof *out, cudaMemcpyDeviceToHost, ctx->stream));
    CRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return CRT_OK;
}

extern "C" int crt_rays_decided_at_emission(crt_ctx* ctx, unsigned long long out[2])
{
    CRT_REQUIRE(ctx && out, "null argument");
    CRT_JOIN_TAIL(ctx);
    out[0] = out[1] = 0;
    if (ctx->queue_counters) CRT_CUDA(cudaMemcpyAsync(out, ctx->queue_counters + 6, sizeof *out, cudaMemcpyDeviceToHost, ctx->stream));
    if (ctx->inline_rays) CRT_CUDA(cudaMemcpyAsync(out + 1, ctx->inline_rays + 2, sizeof *out, cudaMemcpyDeviceToHost, ctx->stream));
    CRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return CRT_OK;
}

template <int EX>
static int path_trace(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom, crt_buffer triangles,
                      crt_buffer lights, crt_raygen raygen, crt_options options, crt_buffer accumulation)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(accumulation, (size_t)W * H, "accumulation");
    CRT_REQUIRE(triangles.data != nullptr, "null triangle buffer");
    CRT_REQUIRE(EX == 7 || bsize(lights) == 0 || lights.data != nullptr, "null light buffer");
    CRT_JOIN_TAIL(ctx);
    unsigned long long* counters = nullptr;
    int rc = inline_ray_counters(ctx, &counters);
    if (rc != CRT_OK) return rc;
    const LightRec* slots = nullptr;  // power-proportional selection: the slot table (uniform: lights[] as the reference)
    uint32_t n_slots = 0;
    if (EX != 7 && ctx->light_mode == CRT_LIGHTS_POWER && bsize(lights))
    {
        CRT_REQUIRE(bsize(lights) < 0xffffffffull, "too many lights");
        rc = light_table_for(ctx, geom, (const float*)triangles.data, (const uint32_t*)lights.data, bsize(lights), &slots, &n_slots);
        if (rc != CRT_OK) return rc;
    }
    // the wavefront form (kernels_paths.cu) packs path | ray << 27 into a record word and keeps a 32-bit visibility mask per vertex
    const bool wave_ok = (size_t)W * H < ((size_t)1 << 27) && (!options.use_shadowed_target_function || options.ris_sample_count <= 32);
    if (ctx->wavefront && wave_ok)
        return path_trace_wavefront(ctx, EX, W, H, frame, geom, (const float*)triangles.data, (const uint32_t*)lights.data,
                                    (uint32_t)bsize(lights), slots, n_slots, raygen, options, (crt_float4*)accumulation.data, counters);
    const Rows rows = rows_of(ctx, H);
    const float* tris60 = (const float*)triangles.data;
    crt_float4* accum = (crt_float4*)accumulation.data;
    with_flag(ctx->math_mode == CRT_MATH_EXACT, [&](auto MODE)
    {
        if (slots)
            k_path_trace<EX, MODE, LightsTable><<<tile_grid(W, rows), 256, 0, ctx->stream>>>(
                W, H, rows, frame, geom->view(), tris60, slots, n_slots, raygen, options, accum, counters);
        else
            k_path_trace<EX, MODE, LightsIndexed><<<tile_grid(W, rows), 256, 0, ctx->stream>>>(
                W, H, rows, frame, geom->view(), tris60, (const uint32_t*)lights.data, (uint32_t)bsize(lights), raygen, options, accum, counters);
    });
    return check_launch(ctx, "path_trace");
}
extern "C" int crt_path_trace_07(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom, crt_buffer triangles,
                                 crt_raygen raygen, crt_options options, crt_buffer accumulation)
{
    return path_trace<7>(ctx, W, H, frame, geom, triangles, crt_buffer{nullptr, 0}, raygen, options, accumulation);
}
extern "C" int crt_path_trace_08(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom, crt_buffer triangles,
                                 crt_buffer lights, crt_raygen raygen, crt_options options, crt_buffer accumulation)
{
    return path_trace<8>(ctx, W, H, frame, geom, triangles, lights, raygen, options, accumulation);
}
extern "C" int crt_path_trace_09(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom, crt_buffer triangles,
                                 crt_buffer lights, crt_raygen raygen, crt_options options, crt_buffer accumulation)
{
    return path_trace<9>(ctx, W, H, frame, geom, triangles, lights, raygen, options, accumulation);
}

extern "C" int crt_ao_06(crt_ctx* ctx, crt_buffer pixels, crt_raygen raygen, int W, int H, crt_geometry geom,
                         crt_buffer triangles, int n_rays)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    CRT_CHECK_IMAGE(W, H);
    CRT_CHECK_BUF(pixels, (size_t)W * H * 4, "pixel");
    CRT_REQUIRE(triangles.data != nullptr, "null triangle buffer");
    CRT_REQUIRE(n_rays > 0, "n_rays must be positive");
    CRT_JOIN_TAIL(ctx);
    unsigned long long* counters = nullptr;
    int rc = inline_ray_counters(ctx, &counters);
    if (rc != CRT_OK) return rc;
    if (ctx->wavefront)
    {
        // bands of rows, so that the ray queue of a band (pixels x n_rays x 32 B) stays below 4 GiB
        const Rows all = rows_of(ctx, H);
        const bool ex = ctx->math_mode == CRT_MATH_EXACT;
        const size_t per_row = (size_t)W * (size_t)n_rays * 32u;
        int band = (int)(((size_t)4 << 30) / (per_row ? per_row : 1));
        band = band < kTileH ? kTileH : band / kTileH * kTileH;
        rc = grow(ctx->ao_count, ctx->ao_count_pixels, (size_t)W * H, (size_t)W * H * sizeof(uint32_t));
        if (rc != CRT_OK) return rc;
        for (int y0 = all.y0; y0 < all.y1; y0 += band)
        {
            const Rows rows{y0, y0 + band < all.y1 ? y0 + band : all.y1};
            const size_t n_px = (size_t)(rows.y1 - rows.y0) * W, n_records = n_px * (size_t)n_rays;
            CRT_REQUIRE(n_records < 0xffffffffull, "too many AO rays in one band");
            ShadowQueue q{nullptr, nullptr, nullptr, 0};
            rc = queue_prepare(ctx, (n_records + 1) / 2, &q);  // capacity is counted in 64-byte records
            if (rc != CRT_OK) return rc;
            q.tmax = kFltMax;  // the reference asks for the closest hit with maxT = FLT_MAX and only uses hit / no hit (:78-82)
            q.stride4 = 2;
            (ex ? k_ao_emit<1> : k_ao_emit<0>)<<<tile_grid(W, rows), 256, 0, ctx->stream>>>(raygen, W, H, rows, geom->view(),
                                                                                         (const float*)triangles.data, n_rays, q,
                                                                                         ctx->ao_count, counters);
            rc = check_launch(ctx, "ao_emit");
            if (rc != CRT_OK) return rc;
            ShadowSink sink{nullptr, nullptr, 0, nullptr};
            sink.visible_count = ctx->ao_count;
            rc = queue_trace<kEpiCountVisible>(ctx, geom, q, sink);
            if (rc != CRT_OK) return rc;
            const size_t first = (size_t)(H - rows.y1) * W;
            (ex ? k_ao_finish<1> : k_ao_finish<0>)<<<sweep_blocks(ctx, n_px), 256, 0, ctx->stream>>>(first, n_px, (uint32_t*)pixels.data,
                                                                                                   ctx->ao_count, n_rays);
            rc = check_launch(ctx, "ao_finish");
            if (rc != CRT_OK) return rc;
        }
        return CRT_OK;
    }
    auto k = ctx->math_mode == CRT_MATH_EXACT ? k_ao<1> : k_ao<0>;
    k<<<tile_grid(W, rows_of(ctx, H)), 256, 0, ctx->stream>>>((uint32_t*)pixels.data, raygen, W, H, rows_of(ctx, H), geom->view(),
                                               (const float*)triangles.data, n_rays, counters);
    return check_launch(ctx, "ao_06");
}
