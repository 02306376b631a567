// api.cu — context, memory, timing and the launch-by-name layer of the C ABI (include/cedecrt.h).
// Replaces the Orochi runtime + common/typedbuffer.hpp + common/shader.hpp of the reference with a thin
// layer over the CUDA runtime: no HIP/CUDA dual dispatch, no run-time compilation, no CPU fallback.
#include <stdlib.h>
#include <string.h>

#include "ctx.cuh"

static_assert(sizeof(crt_triangle) == 60, "Triangle is 60 bytes (common/core.hpp:38-43)");
static_assert(sizeof(crt_visibility) == 16, "Visibility is 16 bytes (common/core.hpp:167-172)");
static_assert(sizeof(crt_reservoir_sample) == 64, "ReservoirSample is 64 bytes (common/reservoir.hpp:5-13)");
static_assert(sizeof(crt_reservoir) == 76, "Reservoir is 76 bytes (common/reservoir.hpp:15-38)");
static_assert(offsetof(crt_reservoir, w_sum) == 64 && offsetof(crt_reservoir, M) == 72, "Reservoir layout");
static_assert(sizeof(crt_options) == 48, "Options is 48 bytes (common/options.hpp:4-23)");
static_assert(offsetof(crt_options, ris_sample_count) == 20 && offsetof(crt_options, use_temporal_resampling) == 28 &&
                  offsetof(crt_options, use_spatial_resampling) == 29 &&
                  offsetof(crt_options, spatial_resampling_sample_count) == 32 &&
                  offsetof(crt_options, use_shadowed_target_function) == 44 &&
                  offsetof(crt_options, use_visibility_reuse) == 45,
              "Options layout");
static_assert(sizeof(crt_raygen) == 36, "RayGenerator is 36 bytes (common/camera.hpp:5-9)");
static_assert(sizeof(crt_buffer) == 16, "TypedBuffer device view is 16 bytes (common/typedbuffer.hpp:14-20)");

using namespace crt;

extern "C" int crt_init(int device, crt_ctx** out)
{
    CRT_REQUIRE(out, "null out pointer");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
    {
        set_error("no CUDA device available (%s); libcedecrt has no CPU path",
                  e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        return CRT_ENODEVICE;
    }
    CRT_REQUIRE(device >= 0 && device < n, "device index out of range");
    CRT_CUDA(cudaSetDevice(device));
    crt_ctx* ctx = new crt_ctx;
    ctx->device = device;
    cudaDeviceProp prop;
    CRT_CUDA(cudaGetDeviceProperties(&prop, device));
    strncpy(ctx->name, prop.name, sizeof ctx->name - 1);
    ctx->sm_count = prop.multiProcessorCount;
    CRT_CUDA(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    CRT_CUDA(cudaEventCreate(&ctx->ev_start));
    CRT_CUDA(cudaEventCreate(&ctx->ev_stop));
    if (const char* e = getenv("CRT_WAVEFRONT")) ctx->wavefront = atoi(e);
    if (const char* e = getenv("CRT_LIGHT_TABLE")) ctx->light_table = atoi(e);
    if (const char* e = getenv("CRT_RESOLVE_REUSE")) ctx->resolve_reuse = atoi(e);
    if (const char* e = getenv("CRT_POOLED_CLOSEST")) ctx->pooled_closest = atoi(e);
    if (const char* e = getenv("CRT_RAYCAST_HINT")) ctx->raycast_hint = atoi(e);
    *out = ctx;
    return CRT_OK;
}

extern "C" int crt_shutdown(crt_ctx* ctx)
{
    if (!ctx) return CRT_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->tail_stream)
    {
        cudaStreamSynchronize(ctx->tail_stream);
        cudaStreamDestroy(ctx->tail_stream);
        cudaEventDestroy(ctx->ev_head);
        cudaEventDestroy(ctx->ev_tail);
    }
    if (ctx->head_stream)
    {
        cudaStreamSynchronize(ctx->head_stream);
        cudaStreamDestroy(ctx->head_stream);
        cudaEventDestroy(ctx->ev_ray_ready);
        cudaEventDestroy(ctx->ev_vis_consumed);
    }
    if (ctx->vis_next) cudaFree(ctx->vis_next);
    if (ctx->queue2_rays) cudaFree(ctx->queue2_rays);
    if (ctx->queue2_counters) cudaFree(ctx->queue2_counters);
    cudaEventDestroy(ctx->ev_start);
    cudaEventDestroy(ctx->ev_stop);
    if (ctx->queue_rays) cudaFree(ctx->queue_rays);
    if (ctx->queue_counters) cudaFree(ctx->queue_counters);
    if (ctx->history_prev) cudaFree(ctx->history_prev);
    if (ctx->tiles) cudaFree(ctx->tiles);
    if (ctx->halo_vis) cudaFree(ctx->halo_vis);
    if (ctx->gbuf) cudaFree(ctx->gbuf);
    if (ctx->inline_rays) cudaFree(ctx->inline_rays);
    if (ctx->ao_count) cudaFree(ctx->ao_count);
    if (ctx->path_state) cudaFree(ctx->path_state);
    for (auto& m : ctx->prof_marks) cudaEventDestroy(m.second);
    for (auto& e : ctx->prof_pool) cudaEventDestroy(e);
    if (ctx->prof_start) cudaEventDestroy(ctx->prof_start);
    cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return CRT_OK;
}

extern "C" const char* crt_device_name(crt_ctx* ctx) { return ctx ? ctx->name : ""; }

extern "C" int crt_set_math_mode(crt_ctx* ctx, int mode)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_REQUIRE(mode == CRT_MATH_LIBDEVICE || mode == CRT_MATH_EXACT || mode == CRT_MATH_FAST || mode == CRT_MATH_REFERENCE,
                "unknown math mode");
    ctx->math_mode = mode;
    return CRT_OK;
}

extern "C" int crt_set_light_sampling(crt_ctx* ctx, int mode, int log2_slots)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_REQUIRE(mode == CRT_LIGHTS_UNIFORM || mode == CRT_LIGHTS_POWER, "unknown light sampling mode");
    CRT_REQUIRE(log2_slots >= 0, "log2_slots must be 0 (the default) or the log2 of the slot count");
    // whether 2^log2_slots fits the light count is checked by the first call that samples lights
    ctx->light_mode = mode;
    ctx->light_log2 = log2_slots;
    return CRT_OK;
}

extern "C" int crt_set_light_tiles(crt_ctx* ctx, int log2_tiles, int log2_tile_size)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_REQUIRE(log2_tiles >= 0 && log2_tiles <= 16, "log2_tiles must be in [0, 16]");
    CRT_REQUIRE(log2_tile_size >= 0 && log2_tile_size <= 16, "log2_tile_size must be in [0, 16]");
    CRT_REQUIRE(log2_tiles + log2_tile_size <= 22, "light tiles hold at most 2^22 records: log2_tiles + log2_tile_size <= 22");
    ctx->tiles_log2_t = log2_tiles;
    ctx->tiles_log2_s = log2_tile_size;
    return CRT_OK;
}

extern "C" int crt_set_reuse_weights(crt_ctx* ctx, int mode)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_REQUIRE(mode == CRT_REUSE_REFERENCE || mode == CRT_REUSE_UNBIASED, "unknown reuse weight mode");
    // the combinations CRT_REUSE_UNBIASED does not cover (a previous camera without surfaces, the fused frame on a row range
    // without crt_restir_set_halo_surfaces) are refused by the calls that would run them
    ctx->reuse_mode = mode;
    return CRT_OK;
}

extern "C" int crt_set_row_range(crt_ctx* ctx, int y_begin, int y_end)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_REQUIRE(y_begin >= 0 && (y_end < 0 || y_end >= y_begin), "bad row range");
    ctx->row_begin = y_begin;
    ctx->row_end = y_end;
    return CRT_OK;
}

extern "C" int crt_set_frame_overlap(crt_ctx* ctx, int on)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_JOIN_TAIL(ctx);
    if (on && !ctx->tail_stream)
    {
        CRT_CUDA(cudaSetDevice(ctx->device));
        CRT_CUDA(cudaStreamCreateWithFlags(&ctx->tail_stream, cudaStreamNonBlocking));
        CRT_CUDA(cudaEventCreateWithFlags(&ctx->ev_head, cudaEventDisableTiming));
        CRT_CUDA(cudaEventCreateWithFlags(&ctx->ev_tail, cudaEventDisableTiming));
    }
    ctx->overlap = on ? 1 : 0;
    return CRT_OK;
}
extern "C" int crt_frame_join(crt_ctx* ctx)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_JOIN_TAIL(ctx);
    return CRT_OK;
}
extern "C" void* crt_get_tail_stream(crt_ctx* ctx) { return ctx ? (void*)ctx->tail_stream : nullptr; }

extern "C" int crt_set_stream(crt_ctx* ctx, void* cuda_stream)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_JOIN_TAIL(ctx);
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return CRT_OK;
}
extern "C" void* crt_get_stream(crt_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
extern "C" unsigned long long crt_launch_count(crt_ctx* ctx) { return ctx ? ctx->launches : 0ull; }
extern "C" int crt_shadow_rays_traced(crt_ctx* ctx, unsigned long long out[2])
{
    CRT_REQUIRE(ctx && out, "null argument");
    CRT_JOIN_TAIL(ctx);
    out[0] = out[1] = 0;
    if (!ctx->queue_counters) return CRT_OK;
    CRT_CUDA(cudaMemcpyAsync(out, ctx->queue_counters + 2, 2 * sizeof *out, cudaMemcpyDeviceToHost, ctx->stream));
    CRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return CRT_OK;
}

extern "C" int crt_malloc(crt_ctx* ctx, size_t bytes, void** out)
{
    CRT_REQUIRE(ctx && out, "null argument");
    CRT_CUDA(cudaSetDevice(ctx->device));
    CRT_CUDA(cudaMalloc(out, bytes ? bytes : 16));
    // zeroed: crt_raycast reads the Visibility record of every pixel before it writes it (the hint of px_raycast_hinted —
    // any content is a valid hint, but memory of the library's own making should not be read uninitialised)
    // On the context's stream and waited for: a plain cudaMemset runs on the legacy default stream, asynchronously for
    // device memory, and the context's non-blocking streams do not order themselves after it — it zeroed the tail of a
    // freshly uploaded triangle array in tests/test_gpu_configs.py (GPU batch 34).
    CRT_CUDA(cudaMemsetAsync(*out, 0, bytes ? bytes : 16, ctx->stream));
    CRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return CRT_OK;
}
extern "C" int crt_free(crt_ctx* ctx, void* p)
{
    CRT_REQUIRE(ctx, "null context");
    if (p) CRT_CUDA(cudaFree(p));
    return CRT_OK;
}
extern "C" int crt_memset(crt_ctx* ctx, void* p, int byte, size_t bytes)
{
    CRT_REQUIRE(ctx && (p || !bytes), "null argument");
    CRT_JOIN_TAIL(ctx);
    if (bytes) CRT_CUDA(cudaMemsetAsync(p, byte, bytes, ctx->stream));
    return CRT_OK;
}
extern "C" int crt_memcpy_h2d(crt_ctx* ctx, void* dst, const void* src, size_t bytes)
{
    CRT_REQUIRE(ctx && ((dst && src) || !bytes), "null argument");
    CRT_JOIN_TAIL(ctx);
    if (!bytes) return CRT_OK;
    CRT_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return CRT_OK;
}
// device to device on the context's stream, ordered like every other copy (after the frame tail in flight); asynchronous
extern "C" int crt_memcpy_d2d(crt_ctx* ctx, void* dst, const void* src, size_t bytes)
{
    CRT_REQUIRE(ctx && ((dst && src) || !bytes), "null argument");
    CRT_JOIN_TAIL(ctx);
    if (!bytes) return CRT_OK;
    CRT_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return CRT_OK;
}
extern "C" int crt_memcpy_d2h(crt_ctx* ctx, void* dst, const void* src, size_t bytes)
{
    CRT_REQUIRE(ctx && ((dst && src) || !bytes), "null argument");
    CRT_JOIN_TAIL(ctx);
    if (!bytes) return CRT_OK;
    CRT_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return CRT_OK;
}
extern "C" int crt_memcpy_d2h_async(crt_ctx* ctx, void* dst, const void* src, size_t bytes)
{
    CRT_REQUIRE(ctx && ((dst && src) || !bytes), "null argument");
    CRT_JOIN_TAIL(ctx);
    if (bytes) CRT_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return CRT_OK;
}
extern "C" int crt_sync(crt_ctx* ctx)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_JOIN_TAIL(ctx);
    CRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return CRT_OK;
}
extern "C" int crt_timer_start(crt_ctx* ctx)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_JOIN_TAIL(ctx);
    CRT_CUDA(cudaEventRecord(ctx->ev_start, ctx->stream));
    return CRT_OK;
}
extern "C" int crt_timer_stop_ms(crt_ctx* ctx, float* ms)
{
    CRT_REQUIRE(ctx && ms, "null argument");
    CRT_JOIN_TAIL(ctx);
    CRT_CUDA(cudaEventRecord(ctx->ev_stop, ctx->stream));
    CRT_CUDA(cudaEventSynchronize(ctx->ev_stop));
    CRT_CUDA(cudaEventElapsedTime(ms, ctx->ev_start, ctx->ev_stop));
    return CRT_OK;
}

// ---- per-kernel device times.  Between begin and end every kernel launch of this context is followed by an
// event on the context's stream; end() synchronises and reports, per launch, the time since the previous event
// (kernels of one stream run back to back, so that is the kernel's duration plus any memset/copy queued before it).
extern "C" int crt_profile_begin(crt_ctx* ctx)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_JOIN_TAIL(ctx);
    if (!ctx->prof_start) CRT_CUDA(cudaEventCreate(&ctx->prof_start));
    for (auto& m : ctx->prof_marks) ctx->prof_pool.push_back(m.second);
    ctx->prof_marks.clear();
    CRT_CUDA(cudaEventRecord(ctx->prof_start, ctx->stream));
    ctx->profiling = true;
    return CRT_OK;
}
extern "C" int crt_profile_end(crt_ctx* ctx, char* names, size_t names_cap, float* ms, int ms_cap, int* count)
{
    CRT_REQUIRE(ctx && names && ms && count, "null argument");
    CRT_JOIN_TAIL(ctx);
    CRT_REQUIRE(ctx->profiling, "crt_profile_begin was not called");
    ctx->profiling = false;
    CRT_CUDA(cudaStreamSynchronize(ctx->stream));
    size_t used = 0;
    int n = 0;
    cudaEvent_t prev = ctx->prof_start;
    if (names_cap) names[0] = 0;
    for (auto& m : ctx->prof_marks)
    {
        const size_t len = strlen(m.first);
        if (n >= ms_cap || used + len + 2 > names_cap) break;
        CRT_CUDA(cudaEventElapsedTime(&ms[n], prev, m.second));
        memcpy(names + used, m.first, len);
        used += len;
        names[used++] = '\n';
        names[used] = 0;
        prev = m.second;
        n++;
    }
    *count = n;
    for (auto& m : ctx->prof_marks) ctx->prof_pool.push_back(m.second);
    ctx->prof_marks.clear();
    return CRT_OK;
}

// RayGenerator::lookat, common/camera.hpp:11-25 — host arithmetic, no contraction (see Makefile)
extern "C" void crt_raygen_lookat(crt_raygen* rg, const float eye[3], const float center[3], const float up[3],
                                  float fovy, int width, int height)
{
    const f3 e{eye[0], eye[1], eye[2]}, c{center[0], center[1], center[2]}, u0{up[0], up[1], up[2]};
    const f3 f = normalize(c - e);
    const f3 s = normalize(cross(f, u0));
    const f3 u = cross(s, f);
    const float tan_y = tanf(fovy * 0.5f);
    const float tan_x = tan_y / (float)height * (float)width;
    const f3 r = s * tan_x, up2 = u * tan_y;
    rg->m_origin = {e.x, e.y, e.z};
    rg->m_right = {r.x, r.y, r.z};
    rg->m_up = {up2.x, up2.y, up2.z};
}

// ---- Shader::launch call shape (common/shader.hpp:179-199)
#define ARG(T, i) (*(const T*)params[i])
extern "C" int crt_launch(crt_ctx* ctx, const char* name, void** params, unsigned, unsigned, unsigned, unsigned,
                          unsigned, unsigned)
{
    CRT_REQUIRE(ctx && name && params, "null argument");
    typedef crt_buffer B;
    if (!strcmp(name, "raycast"))
        return crt_raycast(ctx, ARG(int, 0), ARG(int, 1), ARG(crt_geometry, 2), ARG(B, 3), ARG(crt_raygen, 4), ARG(B, 5));
    if (!strcmp(name, "generate_candidate"))
        return crt_generate_candidate(ctx, ARG(int, 0), ARG(int, 1), ARG(int, 2), ARG(crt_geometry, 3), ARG(B, 4),
                                      ARG(B, 5), ARG(crt_float3, 6), ARG(B, 7), ARG(crt_options, 8), ARG(B, 9));
    if (!strcmp(name, "temporal_resampling"))
        return crt_temporal_resampling(ctx, ARG(int, 0), ARG(int, 1), ARG(int, 2), ARG(crt_geometry, 3), ARG(B, 4),
                                       ARG(B, 5), ARG(crt_float3, 6), ARG(crt_options, 7), ARG(B, 8), ARG(B, 9));
    if (!strcmp(name, "temporal_resampling_reprojected"))
        return crt_temporal_resampling_reprojected(ctx, ARG(int, 0), ARG(int, 1), ARG(int, 2), ARG(crt_geometry, 3), ARG(B, 4),
                                                   ARG(B, 5), ARG(crt_float3, 6), ARG(crt_options, 7), ARG(crt_raygen, 8),
                                                   ARG(B, 9), ARG(B, 10));
    if (!strcmp(name, "temporal_resampling_reprojected_surfaces"))
        return crt_temporal_resampling_reprojected_surfaces(ctx, ARG(int, 0), ARG(int, 1), ARG(int, 2), ARG(crt_geometry, 3),
                                                            ARG(B, 4), ARG(B, 5), ARG(crt_float3, 6), ARG(crt_options, 7),
                                                            ARG(crt_raygen, 8), ARG(B, 9), ARG(B, 10), ARG(B, 11));
    if (!strcmp(name, "temporal_resampling_reprojected_motion"))
        return crt_temporal_resampling_reprojected_motion(ctx, ARG(int, 0), ARG(int, 1), ARG(int, 2), ARG(crt_geometry, 3),
                                                          ARG(B, 4), ARG(B, 5), ARG(crt_float3, 6), ARG(crt_options, 7),
                                                          ARG(crt_raygen, 8), ARG(B, 9), ARG(B, 10), ARG(B, 11), ARG(B, 12));
    if (!strcmp(name, "save_temporal_reservoir"))
        return crt_save_temporal_reservoir(ctx, ARG(int, 0), ARG(int, 1), ARG(B, 2), ARG(B, 3));
    if (!strcmp(name, "spatial_resampling"))
        return crt_spatial_resampling(ctx, ARG(int, 0), ARG(int, 1), ARG(int, 2), ARG(int, 3), ARG(crt_geometry, 4),
                                      ARG(B, 5), ARG(B, 6), ARG(crt_float3, 7), ARG(crt_options, 8), ARG(B, 9),
                                      ARG(B, 10));
    if (!strcmp(name, "resolve"))
        return crt_resolve(ctx, ARG(B, 0), ARG(int, 1), ARG(int, 2), ARG(crt_geometry, 3), ARG(B, 4), ARG(B, 5),
                           ARG(crt_float3, 6), ARG(crt_options, 7), ARG(B, 8));
    if (!strcmp(name, "clear")) return crt_clear(ctx, ARG(B, 0), ARG(int, 1), ARG(int, 2));
    if (!strcmp(name, "tone_mapping")) return crt_tone_mapping(ctx, ARG(B, 0), ARG(B, 1), ARG(int, 2), ARG(int, 3));
    if (!strcmp(name, "path_trace_07"))
        return crt_path_trace_07(ctx, ARG(int, 0), ARG(int, 1), ARG(int, 2), ARG(crt_geometry, 3), ARG(B, 4),
                                 ARG(crt_raygen, 5), ARG(crt_options, 6), ARG(B, 7));
    if (!strcmp(name, "path_trace_08"))
        return crt_path_trace_08(ctx, ARG(int, 0), ARG(int, 1), ARG(int, 2), ARG(crt_geometry, 3), ARG(B, 4), ARG(B, 5),
                                 ARG(crt_raygen, 6), ARG(crt_options, 7), ARG(B, 8));
    if (!strcmp(name, "path_trace_09"))
        return crt_path_trace_09(ctx, ARG(int, 0), ARG(int, 1), ARG(int, 2), ARG(crt_geometry, 3), ARG(B, 4), ARG(B, 5),
                                 ARG(crt_raygen, 6), ARG(crt_options, 7), ARG(B, 8));
    if (!strcmp(name, "ao_06"))
        return crt_ao_06(ctx, ARG(B, 0), ARG(crt_raygen, 1), ARG(int, 2), ARG(int, 3), ARG(crt_geometry, 4), ARG(B, 5),
                         ARG(int, 6));
    set_error("crt_launch: unknown kernel '%s'", name);
    return CRT_EINVAL;
}
