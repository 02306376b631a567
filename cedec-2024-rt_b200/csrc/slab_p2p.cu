// slab_p2p.cu — halo exchange between the row slabs of one node by direct peer stores over NVLink.
//
// New with respect to the reference (single GPU).  Each rank owns image rows [y0, y1) of full-size buffers
// (crt_set_row_range).  The kernels of the fused frame that produce reservoir rows store the kHaloRows boundary
// rows into the neighbours' buffers as well (restir_fast.cuh: HaloPeers — peer pointers obtained with cudaIpc,
// crt_ipc_export / crt_ipc_open), so the bytes cross NVLink/NVSwitch once, from the producing kernel's epilogue,
// overlapped with the rest of that kernel, with no staging buffer and no NCCL launch.  crt_slab_exchange then
//   1. (only with push_rows != 0, e.g. for buffers written by other means) copies the boundary rows with a
//      dedicated kernel;
//   2. raises a monotonically increasing counter in each neighbour's flag slot (release at system scope);
//   3. waits (one spinning thread) until both neighbours have raised this rank's slots to the same count.
// Step 3 is the only synchronisation: a neighbour's flag for stage s also proves that it finished every earlier
// stage, which is exactly what makes the later in-place reuse of the halo rows safe (DESIGN.md section 7).
#include "launch_common.cuh"

namespace crt
{
struct CopySeg
{
    const uint4* src;
    uint4* dst;
    size_t n16;  // 16-byte units
};
struct CopyPlan
{
    CopySeg seg[12];
};
__global__ void __launch_bounds__(256) k_push_halo(CopyPlan plan)
{
    const CopySeg s = plan.seg[blockIdx.y];
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < s.n16; i += (size_t)gridDim.x * blockDim.x)
        s.dst[i] = __ldg(s.src + i);
}
// raise `value` in the neighbours' slots, then wait for them to raise mine.  A neighbour that has not answered after
// kWaitLimitNs (a host that stopped issuing, a slab that failed) must not hang the GPU: the wait gives up and leaves
// the stage number in mine[2], which crt_slab_status reports.
constexpr unsigned long long kWaitLimitNs = 4000000000ull;
__device__ __forceinline__ unsigned long long global_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__global__ void k_signal_wait(unsigned long long* up_slot, unsigned long long* down_slot, volatile unsigned long long* mine,
                              unsigned long long value)
{
    __threadfence_system();
    if (up_slot) atomicExch_system(up_slot, value);
    if (down_slot) atomicExch_system(down_slot, value);
    const unsigned long long t0 = global_ns();
    for (int side = 0; side < 2; side++)
    {
        if (!(side ? down_slot : up_slot)) continue;
        while (mine[side] < value)
        {
            __nanosleep(200);
            if (global_ns() - t0 > kWaitLimitNs)
            {
                mine[2] = value;
                break;
            }
        }
    }
    __threadfence_system();
}
}  // namespace crt

using namespace crt;

extern "C" int crt_ipc_export(crt_ctx* ctx, void* device_ptr, unsigned char handle_out[64])
{
    CRT_REQUIRE(ctx && device_ptr && handle_out, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    cudaIpcMemHandle_t h;
    CRT_CUDA(cudaIpcGetMemHandle(&h, device_ptr));
    memcpy(handle_out, &h, 64);
    return CRT_OK;
}
extern "C" int crt_ipc_open(crt_ctx* ctx, const unsigned char handle[64], void** out)
{
    CRT_REQUIRE(ctx && handle && out, "null argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CRT_CUDA(cudaSetDevice(ctx->device));
    CRT_CUDA(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    return CRT_OK;
}
extern "C" int crt_ipc_close(crt_ctx* ctx, void* peer_ptr)
{
    CRT_REQUIRE(ctx, "null context");
    if (peer_ptr) CRT_CUDA(cudaIpcCloseMemHandle(peer_ptr));
    return CRT_OK;
}

extern "C" int crt_restir_reserve(crt_ctx* ctx, int W, int H, void** class_plane_base)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_CHECK_IMAGE(W, H);
    GBuf g;
    const int rc = ensure_gbuf(ctx, (size_t)W * H, &g);
    if (rc != CRT_OK) return rc;
    if (class_plane_base) *class_plane_base = ctx->gbuf;  // the allocation to export; the plane starts at 24 * capacity
    return CRT_OK;
}

extern "C" int crt_slab_set_links(crt_ctx* ctx, const crt_slab_links* links)
{
    CRT_REQUIRE(ctx, "null context");
    if (!links)
    {
        ctx->links_set = false;
        return CRT_OK;
    }
    CRT_REQUIRE(links->my_flags != nullptr, "null flag buffer");
    // With lazy module loading, the first launch of a kernel loads it, and loading waits for the device to go idle:
    // a slab whose wait kernel is already spinning for a neighbour driven by this same host thread would never see
    // that neighbour's launch.  Every kernel of the frame is therefore loaded now.
    {
        cudaFuncAttributes a;
        CRT_CUDA(cudaFuncGetAttributes(&a, k_signal_wait));
        CRT_CUDA(cudaFuncGetAttributes(&a, k_push_halo));
        int rc = preload_fused_kernels();
        if (rc == CRT_OK) rc = preload_dropin_kernels();
        if (rc != CRT_OK) return rc;
    }
    ctx->links = *links;
    ctx->links_set = true;
    ctx->link_epoch = 0;
    return CRT_OK;
}

extern "C" int crt_slab_status(crt_ctx* ctx, unsigned long long* timed_out_stage)
{
    CRT_REQUIRE(ctx && timed_out_stage, "null argument");
    *timed_out_stage = 0;
    if (!ctx->links_set) return CRT_OK;
    CRT_CUDA(cudaMemcpyAsync(timed_out_stage, (const char*)ctx->links.my_flags + 16, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return CRT_OK;
}

extern "C" int crt_slab_exchange(crt_ctx* ctx, int W, int H, int which, int push_rows, const crt_restir_buffers* b)
{
    const int with_class_plane = push_rows > 1;
    CRT_REQUIRE(ctx && b, "null argument");
    CRT_REQUIRE(ctx->links_set, "crt_slab_set_links has not been called");
    CRT_REQUIRE(which >= 0 && which < 3, "which: 0 temporal, 1 reservoir0, 2 reservoir1");
    CRT_REQUIRE(ctx->frame_fused, "the frame in flight took the per-kernel path (AoS reservoirs): exchange its rows on the host");
    CRT_CHECK_IMAGE(W, H);
    CRT_REQUIRE(W % 16 == 0, "direct halo stores need an image width that is a multiple of 16");
    const Rows rows = rows_of(ctx, H);
    const int halo = kHaloRows;
    const crt_slab_links& L = ctx->links;
    const bool has_up = L.up[which] != nullptr, has_down = L.down[which] != nullptr;
    CRT_REQUIRE(rows.y1 - rows.y0 >= halo || (!has_up && !has_down), "slab thinner than the halo: use the NCCL exchange");
    const size_t n = (size_t)W * H;
    const char* local = (const char*)(which == 0 ? b->temporal.data : which == 1 ? b->reservoir0.data : b->reservoir1.data);
    CopyPlan plan;
    int nseg = 0;
    size_t max16 = 0;
    auto add = [&](const char* src, char* dst, size_t bytes)
    {
        plan.seg[nseg++] = CopySeg{(const uint4*)src, (uint4*)dst, bytes / 16};
        if (bytes / 16 > max16) max16 = bytes / 16;
    };
    auto add_rows = [&](char* peer_base, char* peer_class, int ya, int yb)
    {
        // rows [ya, yb) are the contiguous pixels [(H - yb) * W, (H - ya) * W) of every bottom-up plane
        const size_t first = (size_t)(H - yb) * W, count = (size_t)(yb - ya) * W;
        for (int p = 0; p < kSoaPlanes; p++)
        {
            const size_t e = soa_plane_elem(p), off = soa_plane_offset(p, n) + first * e;
            add(local + off, peer_base + off, count * e);
        }
        if (with_class_plane && peer_class)
        {
            const char* cls = (const char*)ctx->gbuf + ctx->gbuf_pixels * 24;
            add(cls + first, peer_class + first, count);
        }
    };
    CRT_REQUIRE(((size_t)W * halo) % 16 == 0 || !with_class_plane, "class-plane rows must be 16-byte multiples");
    CRT_REQUIRE(!with_class_plane || (ctx->gbuf && ctx->gbuf_pixels == n), "crt_restir_reserve(W, H) must precede the exchange");
    if (push_rows && has_up) add_rows((char*)L.up[which], (char*)L.up[3], rows.y0, rows.y0 + halo);
    if (push_rows && has_down) add_rows((char*)L.down[which], (char*)L.down[3], rows.y1 - halo, rows.y1);
    if (nseg)
    {
        const unsigned bx = (unsigned)((max16 + 255) / 256 < (size_t)ctx->sm_count * 2 ? (max16 + 255) / 256 : (size_t)ctx->sm_count * 2);
        k_push_halo<<<dim3(bx ? bx : 1, nseg), 256, 0, ctx->stream>>>(plan);
        const int rc = check_launch(ctx, "push_halo");
        if (rc != CRT_OK) return rc;
    }
    ctx->link_epoch++;
    k_signal_wait<<<1, 1, 0, ctx->stream>>>((unsigned long long*)(has_up ? L.up_flag : nullptr),
                                           (unsigned long long*)(has_down ? L.down_flag : nullptr),
                                           (volatile unsigned long long*)L.my_flags, ctx->link_epoch);
    return check_launch(ctx, "signal_wait");
}
