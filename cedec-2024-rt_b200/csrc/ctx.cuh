// ctx.cuh — context object, error plumbing and launch helpers behind the C ABI (include/cedecrt.h).
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>

#include <string>
#include <utility>
#include <vector>

#include "../../include/cedecrt.h"
#include "bvh.cuh"

struct crt_ctx
{
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;  // the stream every launch and copy goes to
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
    int math_mode = CRT_MATH_REFERENCE;
    int sm_count = 0;
    char name[256] = {0};
    // wavefront shadow rays (shadow_queue.cuh): ray queue + {count, next} counters, grown on demand
    void* queue_rays = nullptr;
    unsigned* queue_counters = nullptr;
    size_t queue_capacity = 0;
    int raycast_hint = 1;  // primary rays seeded with the triangle the pixel's Visibility record names before the call (CRT_RAYCAST_HINT=0: off)
    const void* hint_tris = nullptr;  // the triangle array a crt_raycast of this context has seen to be the tree's own (licence for the prefetch's hints)
    int pooled_closest = 1;  // examples 07-09: closest hits through the persistent pooled kernel (CRT_POOLED_CLOSEST: 0 never, 1 bounce rays, 2 all)
    void* path_state = nullptr;  // examples 07-09 as a wavefront: per-path state (kernels_paths.cu)
    size_t path_state_pixels = 0;
    uint32_t* ao_count = nullptr;  // 06_ao as a wavefront: unoccluded AO rays per pixel
    size_t ao_count_pixels = 0;
    unsigned long long* inline_rays = nullptr;  // {closest-hit, shadow / AO} rays traced by the single-kernel examples 06-09
    // frame overlap (crt_set_frame_overlap): the tail of the fused frame — the resolve rays and tone mapping — runs on a
    // second stream, so that the next frame's raycast and candidate kernels fill the tail's drain (and vice versa)
    int overlap = 0;
    cudaStream_t tail_stream = nullptr;
    cudaEvent_t ev_head = nullptr, ev_tail = nullptr;
    bool tail_pending = false;  // a tail has been issued that ctx->stream has not been ordered after yet
    // the next frame's primary rays ahead of time (crt_restir_prefetch_raycast): a third stream and a second Visibility buffer
    cudaStream_t head_stream = nullptr;
    cudaEvent_t ev_ray_ready = nullptr, ev_vis_consumed = nullptr;
    void* vis_next = nullptr;
    size_t vis_next_pixels = 0;
    bool ray_next_valid = false, vis_consumed_pending = false;
    crt_raygen ray_next_cam = {};
    unsigned long long ray_next_geom = 0;
    int ray_next_dims[4] = {0, 0, 0, 0};  // W, H, y0, y1
    void* queue2_rays = nullptr;  // the resolve rays' own queue while frames overlap (the next frame's visibility-reuse rays use the first)
    unsigned* queue2_counters = nullptr;
    size_t queue2_capacity = 0;
    int wavefront = 1;  // 0: trace shadow rays inside the per-pixel kernels (CRT_WAVEFRONT=0)
    int light_table = 1;  // 0: sample lights through lights[] -> triangles[] like the reference (CRT_LIGHT_TABLE=0; uniform mode only)
    int light_mode = CRT_LIGHTS_UNIFORM;  // crt_set_light_sampling
    int light_log2 = 0;                   // requested log2 of the slot count of CRT_LIGHTS_POWER; 0: the default
    // presampled light tiles of the ReSTIR DI candidates (crt_set_light_tiles; both 0: off) and the buffer of the last
    // build, valid for (geometry serial, source table generation, frame, log2 T, log2 S) = tiles_key
    int tiles_log2_t = 0, tiles_log2_s = 0;
    void* tiles = nullptr;
    size_t tiles_cap = 0;  // records the allocation holds
    bool tiles_valid = false;
    unsigned long long tiles_key[5] = {0, 0, 0, 0, 0};
    int reuse_mode = CRT_REUSE_REFERENCE;  // crt_set_reuse_weights
    // fused frame (kernels_fast.cu): G-buffer + pixel-class plane, 25 bytes per pixel, grown on demand
    void* gbuf = nullptr;
    size_t gbuf_pixels = 0;
    // traced marks of the temporal history (restir_fast.cuh: kTracedBit) are valid for this geometry and buffer
    unsigned long long history_serial = 0;
    const void* history_buffer = nullptr;
    // temporal reprojection in the fused frame (crt_restir_set_previous_camera): the previous frame's camera and a snapshot
    // of its history (the merge of the fused frame is in place, a look-up at another pixel must not see this frame's records)
    bool prev_cam_set = false;
    crt_raygen prev_cam = {};
    // the previous frame's Visibility buffer (crt_restir_set_previous_frame; data == nullptr: not given): the history
    // pixel's surface for CRT_REUSE_UNBIASED
    crt_buffer prev_vis = {};
    // the previous frame's triangle array (crt_restir_set_previous_triangles; data == nullptr: the geometry did not move),
    // read with a previous camera only
    crt_buffer prev_tris = {};
    void* history_prev = nullptr;
    size_t history_prev_pixels = 0;
    // CRT_REUSE_UNBIASED in the fused frame on a row range (crt_restir_set_halo_surfaces): the G-buffer records of the rows
    // the spatial passes read beyond the range, from primary rays traced into a Visibility buffer of the context's own
    int halo_surfaces = 0;
    void* halo_vis = nullptr;      // two bands of h * W records (kernels_fast.cu: halo_surfaces)
    size_t halo_vis_pixels = 0;    // records allocated
    int halo_reach = 0;            // rows on each side of the range the last crt_restir_frame_begin covered (0: none)
    int halo_dims[2] = {0, 0};     // and the image size it covered them for
    int resolve_reuse = 1;  // 0: resolve traces every shadow ray like the reference (CRT_RESOLVE_REUSE=0)
    // slab_p2p.cu: peer pointers of the neighbouring slabs and the exchange counter
    crt_slab_links links = {};
    bool links_set = false;
    bool frame_fused = true;  // the last crt_restir_frame_begin ran the fused bodies (SoA reservoirs), not the per-kernel path
    unsigned long long link_epoch = 0;
    int row_begin = 0, row_end = -1;  // rows of yi this context computes (crt_set_row_range); -1 = image height
    unsigned long long launches = 0;  // kernels launched through this context (bench.py: gpu_launches)
    // crt_profile_begin/end: an event after every launch; consecutive differences are per-kernel device times
    bool profiling = false;
    cudaEvent_t prof_start = nullptr;
    std::vector<std::pair<const char*, cudaEvent_t>> prof_marks;
    std::vector<cudaEvent_t> prof_pool;
};

struct crt_geometry_t
{
    crt::WideNode* nodes = nullptr;
    crt::WideTri* tris = nullptr;
    const crt_triangle* src = nullptr;  // the triangle array the tree was built over
    size_t n_tris = 0, n_nodes = 0;
    unsigned long long serial = 0;  // unique per build, never 0 (crt_ctx::history_serial)
    int max_depth = 0;
    float build_ms = 0.0f;
    float pad = 0.0f;
    int device = 0;
    // 64-byte light records (restir_core.cuh: LightRec) for the light list last seen by a light-sampling kernel: one per
    // light, or one per slot of power-proportional selection (light_table_log2 = log2 K; -1: uniform)
    void* light_table = nullptr;
    const void* light_table_key = nullptr;
    size_t light_table_n = 0;
    size_t light_table_cap = 0;  // records the allocation holds
    int light_table_log2 = -1;
    unsigned long long light_table_gen = 0;  // counts the rebuilds of light_table (the key of a context's light tiles)
    void* light_scratch = nullptr;  // the slot table's build scratch (geometry.cu: build_light_slots), grown on demand
    size_t light_scratch_bytes = 0;
    float postpone_ratio = crt::kPostponeRatio;
    // refit (crt_refit_geometry): first node of every level of the wide tree, exact node boxes (allocated on demand)
    std::vector<uint32_t> level_begin;
    float* node_box = nullptr;
    float refit_ms = 0.0f;
    crt::Bvh view() const { return crt::Bvh{nodes, tris, postpone_ratio}; }
};

namespace crt
{
void set_error(const char* fmt, ...);

#define CRT_CUDA(call)                                                                        \
    do                                                                                        \
    {                                                                                         \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess)                                                               \
        {                                                                                     \
            crt::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return e__ == cudaErrorMemoryAllocation ? CRT_ENOMEM : CRT_ECUDA;                 \
        }                                                                                     \
    } while (0)

#define CRT_REQUIRE(cond, msg)                          \
    do                                                  \
    {                                                   \
        if (!(cond))                                    \
        {                                               \
            crt::set_error("%s: %s", __func__, (msg));  \
            return CRT_EINVAL;                          \
        }                                               \
    } while (0)

inline int check_launch(crt_ctx* ctx, const char* what, cudaStream_t on = nullptr)
{
    ctx->launches++;
    if (ctx->profiling)
    {
        cudaEvent_t ev = nullptr;
        if (!ctx->prof_pool.empty())
        {
            ev = ctx->prof_pool.back();
            ctx->prof_pool.pop_back();
        }
        else cudaEventCreate(&ev);
        cudaEventRecord(ev, on ? on : ctx->stream);
        ctx->prof_marks.emplace_back(what, ev);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
    {
        set_error("launch of %s failed: %s", what, cudaGetErrorString(e));
        return CRT_ECUDA;
    }
    return CRT_OK;
}

// order everything issued to ctx->stream from now on after the frame tail in flight (no-op without overlap)
inline int join_tail(crt_ctx* ctx)
{
    if (ctx->tail_pending)
    {
        CRT_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_tail, 0));
        ctx->tail_pending = false;
    }
    return CRT_OK;
}
#define CRT_JOIN_TAIL(ctx)                        \
    do                                            \
    {                                             \
        const int rc__ = crt::join_tail(ctx);     \
        if (rc__ != CRT_OK) return rc__;          \
    } while (0)

inline unsigned div_up(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

// device memory grown on demand: when the capacity `cap` (in the caller's unit) is below `want`, the buffer is replaced by
// one of `bytes` bytes.  Pointer and capacity are cleared before the allocation, so a failed cudaMalloc leaves an empty,
// consistent buffer.  *fresh tells whether the memory is new (its contents undefined): each caller fills it on its own stream.
template <class T>
int grow(T*& p, size_t& cap, size_t want, size_t bytes, bool* fresh = nullptr)
{
    if (fresh) *fresh = false;
    if (cap >= want) return CRT_OK;
    if (p) CRT_CUDA(cudaFree(p));
    p = nullptr;
    cap = 0;
    CRT_CUDA(cudaMalloc((void**)&p, bytes));
    cap = want;
    if (fresh) *fresh = true;
    return CRT_OK;
}
}  // namespace crt
