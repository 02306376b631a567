// kernels_fast.cu — the fused ReSTIR DI frame ("fast mode"): crt_restir_di_frame and its staged form.
//
// One call replaces the launch list of examples/10_restir_di/10_restir_di.cpp:270-372.  The per-pixel bodies are
// in restir_fast.cuh (what is fused and why); this file holds the kernels and the frame schedule:
//
//   k_raycast                    primary visibility                         (10_restir_di.cu:9-34)
//   k_candidate_temporal         RIS candidates + temporal merge, in place  (:36-237, save_temporal :239-254 vanishes)
//   k_trace_shadow_queue<2>      visibility-reuse rays of surviving candidates only
//   k_spatial_fast  x passes     temporal -> reservoir1 -> reservoir0 -> reservoir1 ...   (:256-388)
//   k_resolve_fast               sky/emissive pixels finished, shading factors + ray queued (:390-459)
//   k_trace_shadow_queue<1>      resolve rays; accumulation written in the epilogue
//   k_tone_mapping               (crt_tone_mapping, common.cu:30-74)
//
// Buffer roles (all planar SoA, restir_fast.cuh: SoaStore, inside the caller's TypedBuffer<Reservoir> storage):
// `temporal` is read (last frame) and rewritten (this frame) in place; spatial pass 0 reads it and writes
// reservoir1, later passes ping-pong reservoir1 <-> reservoir0, so the final reservoirs are where the reference
// leaves them (reservoir1 for an odd pass count, reservoir0 for an even one).
//
// Options the fused bodies do not cover (use_shadowed_target_function: rays inside the target function) run the
// per-kernel path of kernels_dropin.cu on AoS buffers instead — same results, reference data flow.
#include "launch_common.cuh"

// This file is compiled three times (csrc/Makefile).  The regular object carries the host API and the per-pixel kernels
// in namespace crt::ex, compiled like the rest of the library (-fmad=false, IEEE division and square root: the
// arithmetic the CPU oracle checks bit for bit; CRT_MATH_LIBDEVICE and CRT_MATH_EXACT).  The other two carry only the
// per-pixel kernels again:
//   crt::rf  -DCRT_REFMATH_TU   -fmad=true, IEEE division / square root, libdevice functions — nvcc's and NVRTC's
//                               defaults, i.e. the arithmetic of the reference's own GPU build (10_restir_di.cpp:56-70
//                               passes no floating-point option): CRT_MATH_REFERENCE, the default mode;
//   crt::fm  -DCRT_FASTMATH_TU  -use_fast_math: CRT_MATH_FAST.
// Traversal and the triangle test are not in these kernels (shadow rays are queued, primary rays are k_raycast), so
// they stay exact in every mode.
#if defined(CRT_FASTMATH_TU)
#define CRT_KNS fm
#define CRT_AUX_TU 1
#elif defined(CRT_REFMATH_TU)
#define CRT_KNS rf
#define CRT_AUX_TU 1
#else
#define CRT_KNS ex
#endif

namespace crt
{
// the host-side launchers of the fused frame's per-pixel kernels; each of ex, rf and fm defines one set, kLaunchers
struct FusedLaunchers
{
    int (*preload)();
    void (*candidate_temporal)(cudaStream_t st, bool exact, dim3 grid, int W, int H, Rows rows, int frame, Bvh bvh,
                               const float* tris60, const crt_visibility* vis, f3 eye, const LightRec* table,
                               const uint32_t* light_ids, uint32_t n_lights, crt_options options, SoaStore T, GBuf g,
                               ShadowQueue q, HaloPeers peers, const Reprojection* rp, int reuse, const LightsTiles* tiles,
                               const float* prev_tris60);
    void (*spatial)(cudaStream_t st, bool exact, dim3 grid, int W, int H, Rows rows, int frame, int pass, Bvh bvh, f3 eye,
                    crt_options options, SoaStore in, SoaStore out, GBuf g, HaloPeers peers, int reuse);
    void (*resolve)(cudaStream_t st, dim3 grid, crt_float4* accum, int W, int H, Rows rows, const float* tris60,
                    const crt_visibility* vis, SoaStore res, GBuf g, ShadowQueue q, int accumulate, int reuse_traced);
    void (*halo_surfaces)(cudaStream_t st, dim3 grid, int W, int H, Rows rows, const float* tris60, const crt_visibility* vis,
                          f3 eye, GBuf g);
};
namespace CRT_KNS
{
#ifndef CRT_CT_MINBLOCKS
#define CRT_CT_MINBLOCKS 3  // 80 registers; measured best with kRisBatch = 2 (profiles/r1/tuning_j.txt)
#endif
// RW: the reuse weights of the temporal merge (crt_set_reuse_weights), CRT_REUSE_REFERENCE or CRT_REUSE_UNBIASED
template <class L, int MODE, int RW>
__global__ void __launch_bounds__(256, CRT_CT_MINBLOCKS)
    k_candidate_temporal(int W, int H, Rows rows, int frame, Bvh bvh, const float* tris60, const crt_visibility* vis, f3 eye,
                         L lights, crt_options options, SoaStore temporal, GBuf g, ShadowQueue q, HaloPeers peers)
{
    const TilePix t = this_pixel(W, H, rows);
    DeferredRay d{false, {0, 0, 0}, {0, 0, 0}};
    CandPixel cp{Vis{0.0f, 0.0f, -1}, true};
    if (t.in) cp = classify_pixel(t.px, tris60, vis);
    // lanes 2k, 2k+1 are horizontal neighbours of the warp's 8x4 tile: they share their light-record gathers
    const unsigned pairs = complete_pairs(__ballot_sync(0xffffffffu, t.in && !cp.skip));
    if (t.in) d = px_candidate_temporal<Math<MODE>, L, false, RW>(t.px, cp, frame, bvh, tris60, eye, lights, make_opt(options), temporal, g, peers, pairs);
    queue_push(q, d.want, to_shadow_ray(d, t.px.idx), d.decided);
}
// the same with temporal reprojection (px_candidate_temporal<..., REPROJ = true>); a kernel of its own so that the
// in-place kernel above keeps its registers and its code.  RW = CRT_REUSE_UNBIASED reads rp.prev_vis at the history pixel.
// MOTION: moving geometry, `prev_tris60` is the previous frame's triangle array (crt_restir_set_previous_triangles); the
// other instantiations ignore it (the last parameter, so that they keep their code)
template <class L, int MODE, int RW, bool MOTION = false>
__global__ void __launch_bounds__(256, CRT_CT_MINBLOCKS)
    k_candidate_temporal_reprojected(int W, int H, Rows rows, int frame, Bvh bvh, const float* tris60, const crt_visibility* vis, f3 eye,
                                     L lights, crt_options options, SoaStore temporal, GBuf g, ShadowQueue q, HaloPeers peers, Reprojection rp,
                                     const float* prev_tris60)
{
    const TilePix t = this_pixel(W, H, rows);
    DeferredRay d{false, {0, 0, 0}, {0, 0, 0}};
    CandPixel cp{Vis{0.0f, 0.0f, -1}, true};
    if (t.in) cp = classify_pixel(t.px, tris60, vis);
    if (t.in)
        d = px_candidate_temporal<Math<MODE>, L, true, RW, MOTION>(t.px, cp, frame, bvh, tris60, eye, lights, make_opt(options),
                                                                   temporal, g, peers, 0u, rp, prev_tris60);
    queue_push(q, d.want, to_shadow_ray(d, t.px.idx), d.decided);
}
#ifndef CRT_SP_MINBLOCKS
#define CRT_SP_MINBLOCKS 4  // 64 registers: 0.83 -> 0.75 ms per pass against 3 (profiles/r1/tuning_q.txt)
#endif
template <int MODE, int RW>
__global__ void __launch_bounds__(256, CRT_SP_MINBLOCKS)
    k_spatial_fast(int W, int H, Rows rows, int frame, int pass, Bvh bvh, f3 eye, crt_options options, SoaStore in,
                   SoaStore out, GBuf g, HaloPeers peers)
{
    const TilePix t = this_pixel(W, H, rows);
    if (t.in) px_spatial_fast<Math<MODE>, RW>(t.px, W, H, frame, pass, bvh, eye, make_opt(options), in, out, g, peers);
}
__global__ void __launch_bounds__(256)
    k_resolve_fast(crt_float4* accum, int W, int H, Rows rows, const float* tris60,
                   const crt_visibility* vis, SoaStore res, GBuf g, ShadowQueue q, int accumulate, int reuse_traced)
{
    const TilePix t = this_pixel(W, H, rows);
    DeferredRay d{false, {0, 0, 0}, {0, 0, 0}};
    DeferredShade sh{{0, 0, 0}, {0, 0, 0}, 0.0f};
    if (t.in) d = px_resolve_fast(t.px, accum, tris60, vis, res, g, sh, accumulate != 0, reuse_traced != 0);
    ShadowRay r = to_shadow_ray(d, t.px.idx);
    r.ucw = sh.ucw;
    r.bgx = sh.bg.x; r.bgy = sh.bg.y; r.bgz = sh.bg.z;
    r.rx = sh.rad.x; r.ry = sh.rad.y; r.rz = sh.rad.z;
    // one atomic per block: 0.370 -> 0.255 ms at 4K (per warp, the appends were one same-address atomic every 1.4 ns — the
    // L2's limit; in k_candidate_temporal, 2 ms long, the per-warp form is the faster one: 2.035 against 2.086 ms)
    queue_push_block(q, d.want, r);
}
// G-buffer records of halo rows (crt_restir_set_halo_surfaces) from the context's own Visibility of those rows
__global__ void __launch_bounds__(256)
    k_halo_surfaces(int W, int H, Rows rows, const float* tris60, const crt_visibility* vis, f3 eye, GBuf g)
{
    const TilePix t = this_pixel(W, H, rows);
    if (t.in) px_halo_surface(t.px, tris60, vis, eye, g);
}

// host-side launchers, one set per namespace (the API below picks the set of the context's math mode: FusedLaunchers)
void launch_candidate_temporal(cudaStream_t st, bool exact, dim3 grid, int W, int H, Rows rows, int frame, Bvh bvh,
                               const float* tris60, const crt_visibility* vis, f3 eye, const LightRec* table,
                               const uint32_t* light_ids, uint32_t n_lights, crt_options options, SoaStore T, GBuf g,
                               ShadowQueue q, HaloPeers peers, const Reprojection* rp, int reuse, const LightsTiles* tiles,
                               const float* prev_tris60)
{
    auto launch = [&](auto L)
    {
        with_math_reuse(exact, reuse, [&](auto MODE, auto RW)
        {
            if (rp)
                with_flag(prev_tris60 != nullptr, [&](auto MOTION)
                {
                    k_candidate_temporal_reprojected<decltype(L), MODE, RW, MOTION><<<grid, 256, 0, st>>>(
                        W, H, rows, frame, bvh, tris60, vis, eye, L, options, T, g, q, peers, *rp, prev_tris60);
                });
            else k_candidate_temporal<decltype(L), MODE, RW><<<grid, 256, 0, st>>>(W, H, rows, frame, bvh, tris60, vis, eye, L, options, T, g, q, peers);
        });
    };
    if (tiles) launch(*tiles);  // crt_set_light_tiles: the candidates draw from the pixel's tile of this frame
    else if (table) launch(LightsTable{table, n_lights});
    else launch(LightsIndexed{tris60, light_ids, n_lights});
}
void launch_spatial(cudaStream_t st, bool exact, dim3 grid, int W, int H, Rows rows, int frame, int pass, Bvh bvh, f3 eye,
                    crt_options options, SoaStore in, SoaStore out, GBuf g, HaloPeers peers, int reuse)
{
    with_math_reuse(exact, reuse, [&](auto MODE, auto RW)
                    { k_spatial_fast<MODE, RW><<<grid, 256, 0, st>>>(W, H, rows, frame, pass, bvh, eye, options, in, out, g, peers); });
}
void launch_resolve(cudaStream_t st, dim3 grid, crt_float4* accum, int W, int H, Rows rows, const float* tris60,
                    const crt_visibility* vis, SoaStore res, GBuf g, ShadowQueue q, int accumulate, int reuse_traced)
{
    k_resolve_fast<<<grid, 256, 0, st>>>(accum, W, H, rows, tris60, vis, res, g, q, accumulate, reuse_traced);
}
void launch_halo_surfaces(cudaStream_t st, dim3 grid, int W, int H, Rows rows, const float* tris60, const crt_visibility* vis,
                          f3 eye, GBuf g)
{
    k_halo_surfaces<<<grid, 256, 0, st>>>(W, H, rows, tris60, vis, eye, g);
}
int preload()
{
    cudaFuncAttributes a;
    // both reuse weights and every light source: CRT_REUSE_UNBIASED (with halo surfaces, crt_restir_set_halo_surfaces) and
    // light tiles run over slab links too.  The reprojected candidate kernels are not loaded: reprojection does not run over
    // slab links.
    for (int exact = 0; exact < 2; exact++)
        for (int reuse : {CRT_REUSE_REFERENCE, CRT_REUSE_UNBIASED})
        {
            const int rc = with_math_reuse(exact, reuse, [&](auto MODE, auto RW) -> int
            {
                CRT_CUDA(cudaFuncGetAttributes(&a, k_candidate_temporal<LightsTable, MODE, RW>));
                CRT_CUDA(cudaFuncGetAttributes(&a, k_candidate_temporal<LightsIndexed, MODE, RW>));
                CRT_CUDA(cudaFuncGetAttributes(&a, k_candidate_temporal<LightsTiles, MODE, RW>));
                CRT_CUDA(cudaFuncGetAttributes(&a, k_spatial_fast<MODE, RW>));
                return CRT_OK;
            });
            if (rc != CRT_OK) return rc;
        }
    CRT_CUDA(cudaFuncGetAttributes(&a, k_resolve_fast));
    CRT_CUDA(cudaFuncGetAttributes(&a, k_halo_surfaces));
    return CRT_OK;
}
extern const FusedLaunchers kLaunchers = {preload, launch_candidate_temporal, launch_spatial, launch_resolve, launch_halo_surfaces};
}  // namespace CRT_KNS

#if !defined(CRT_AUX_TU)
namespace fm
{
extern const FusedLaunchers kLaunchers;
}
namespace rf
{
extern const FusedLaunchers kLaunchers;
}
// the launchers whose kernels implement the context's math mode
static const FusedLaunchers& launchers(const crt_ctx* ctx)
{
    return ctx->math_mode == CRT_MATH_FAST ? fm::kLaunchers : ctx->math_mode == CRT_MATH_REFERENCE ? rf::kLaunchers : ex::kLaunchers;
}
// the traced marks of a history buffer stop being true when the geometry they were traced against is replaced
// Only this context's own rows (pixels [first, first + n) of the bottom-up buffer): with slab links set, the halo rows
// of the buffer are stored into by the neighbours' kernels — and rewritten by them in full every frame, marks included —
// so a read-modify-write from here would race with those stores for nothing.
__global__ void __launch_bounds__(256) k_clear_traced(size_t first, size_t n, SoaStore s)
{
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (size_t)gridDim.x * blockDim.x)
    {
        const size_t i = first + k;
        uint32_t* w = s.mword((int)i);
        const uint32_t v = *w;
        if (v & kTracedBit) *w = v & ~kTracedBit;
    }
}
int preload_fused_kernels()
{
    cudaFuncAttributes a;
    CRT_CUDA(cudaFuncGetAttributes(&a, k_clear_traced));
    CRT_CUDA(cudaFuncGetAttributes(&a, k_trace_shadow_queue<kEpiSoaVisibility>));
    CRT_CUDA(cudaFuncGetAttributes(&a, k_trace_shadow_queue<kEpiResolve>));
    CRT_CUDA(cudaFuncGetAttributes(&a, k_build_light_table));
    int rc = ex::kLaunchers.preload();
    if (rc == CRT_OK) rc = rf::kLaunchers.preload();
    return rc != CRT_OK ? rc : fm::kLaunchers.preload();
}
// layout conversion for inspection / parity dumps / switching modes with history
__global__ void __launch_bounds__(256) k_soa_to_aos(size_t n, SoaStore s, crt_reservoir* aos)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) soa_to_aos(s, aos, (int)i);
}
__global__ void __launch_bounds__(256) k_aos_to_soa(size_t n, const crt_reservoir* aos, SoaStore s)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) aos_to_soa(aos, s, (int)i);
}
#endif  // !CRT_AUX_TU (the namespace closes in every build)
}  // namespace crt

#if !defined(CRT_AUX_TU)
using namespace crt;

int crt::ensure_gbuf(crt_ctx* ctx, size_t n, GBuf* g)
{
    bool fresh = false;
    const int rc = grow(ctx->gbuf, ctx->gbuf_pixels, n, n * 25 + 256, &fresh);
    if (rc != CRT_OK) return rc;
    if (fresh) CRT_CUDA(cudaMemsetAsync(ctx->gbuf, 0, n * 25 + 256, ctx->stream));
    const size_t cap = ctx->gbuf_pixels;
    g->g0 = (char*)ctx->gbuf;
    g->g1 = g->g0 + cap * 16;
    g->cls = (uint8_t*)(g->g1 + cap * 8);
    return CRT_OK;
}

namespace
{
// The fused bodies cover every option set except rays inside the target function; M must fit the 29 bits the
// record gives it: (M-cap + candidates) x (neighbours + 1)^passes (10_restir_di.cu:186-188, reservoir.hpp:31-37).
bool fused(const crt_options& o)
{
    if (o.use_shadowed_target_function) return false;
    double m = 21.0 * (o.ris_sample_count > 0 ? o.ris_sample_count : 0);
    if (o.use_spatial_resampling)
        for (int p = 0; p < o.spatial_resampling_passes && m < 1e12; p++)
            m *= 1.0 + (o.spatial_resampling_sample_count > 0 ? o.spatial_resampling_sample_count : 0);
    return m < (double)kMMask;
}
SoaStore soa(const crt_buffer& b, size_t n) { return SoaStore{(char*)b.data, n}; }
int check_buffers(int W, int H, const crt_restir_buffers* b)
{
    CRT_REQUIRE(b, "null buffer set");
    CRT_CHECK_IMAGE(W, H);
    const size_t n = (size_t)W * H;
    CRT_CHECK_BUF(b->pixels, n * 4, "pixel");
    CRT_CHECK_BUF(b->accumulation, n, "accumulation");
    CRT_CHECK_BUF(b->visibility, n, "visibility");
    CRT_CHECK_BUF(b->reservoir0, n, "reservoir0");
    CRT_CHECK_BUF(b->reservoir1, n, "reservoir1");
    CRT_CHECK_BUF(b->temporal, n, "temporal reservoir");
    CRT_REQUIRE(b->reservoir0.data != b->reservoir1.data && b->reservoir0.data != b->temporal.data &&
                    b->reservoir1.data != b->temporal.data,
                "the three reservoir buffers must be distinct");
    return CRT_OK;
}
// the neighbours' copies of reservoir buffer `which` (0 temporal, 1 reservoir0, 2 reservoir1) for kernels that
// mirror their boundary rows (crt_slab_set_links with slabs at least kHaloRows tall); empty otherwise
HaloPeers halo_peers(const crt_ctx* ctx, int which, Rows rows, bool with_class, size_t n)
{
    HaloPeers p;
    if (!ctx->links_set || rows.y1 - rows.y0 < kHaloRows) return p;
    p.up = (char*)ctx->links.up[which];
    p.down = (char*)ctx->links.down[which];
    if (with_class)
    {
        p.up_cls = (uint8_t*)ctx->links.up[3];
        p.down_cls = (uint8_t*)ctx->links.down[3];
    }
    p.up_end = rows.y0 + kHaloRows;
    p.down_begin = rows.y1 - kHaloRows;
    (void)n;
    return p;
}
// the fused spatial pass of CRT_REUSE_UNBIASED reads its neighbours' G-buffer records, which the candidate kernel writes for
// this context's own rows only: it runs on the whole image and without slab links, unless the context produces the records
// of its halo rows itself (crt_restir_set_halo_surfaces)
bool whole_image(const crt_ctx* ctx, int H)
{
    const Rows rows = rows_of(ctx, H);
    return rows.y0 == 0 && rows.y1 == H && !ctx->links_set;
}
bool unbiased_rows_ok(const crt_ctx* ctx, int H, const crt_options& o) { return !fused(o) || whole_image(ctx, H) || ctx->halo_surfaces; }
const char* const kUnbiasedRowsMsg = "unbiased reuse weights in the fused frame need the whole image on one context (no row "
                                     "range, no slab links) or crt_restir_set_halo_surfaces: the G-buffer of halo rows is not "
                                     "kept otherwise; the per-kernel path takes row ranges";
const char* const kHaloReachMsg = "the halo surfaces of crt_restir_frame_begin do not reach as far as this spatial pass's "
                                  "spatial_resampling_radius (or were made for another image size): begin the frame with the "
                                  "options of its spatial passes";
// CRT_REUSE_UNBIASED on a row range (crt_restir_set_halo_surfaces): the G-buffer records of rows [y0 - h, y0) and
// [y1, y1 + h), clipped to the image, h = halo_rows_for(radius) — every row this frame's spatial passes can read beyond
// the range.  Primary rays into a Visibility buffer of the context's own (the host's buffer rows outside the range belong
// to other contexts or to an NCCL receive), then the surface of every diffuse pixel (px_halo_surface).  Records the reach
// for crt_restir_spatial_pass.  Nothing is launched under CRT_REUSE_REFERENCE, without spatial passes, on the whole image.
int halo_surfaces(crt_ctx* ctx, int W, int H, crt_geometry geom, const float* tris60, crt_raygen raygen, f3 eye,
                  const crt_options& o, Rows rows, const GBuf& g)
{
    ctx->halo_reach = 0;
    if (!ctx->halo_surfaces || ctx->reuse_mode != CRT_REUSE_UNBIASED || !o.use_spatial_resampling || o.spatial_resampling_passes <= 0)
        return CRT_OK;
    const int h = halo_rows_for(o.spatial_resampling_radius);
    const Rows bands[2] = {{rows.y0 - h > 0 ? rows.y0 - h : 0, rows.y0}, {rows.y1, rows.y1 + h < H ? rows.y1 + h : H}};
    // the Visibility records of the two bands only: h rows of W records each, band k at record k * h * W
    const size_t band_cap = (size_t)h * W;
    for (int k = 0; k < 2; k++)
    {
        const Rows& b = bands[k];
        if (b.y1 <= b.y0 || rows.y1 <= rows.y0) continue;
        bool fresh = false;
        int rc = grow(ctx->halo_vis, ctx->halo_vis_pixels, 2 * band_cap, 2 * band_cap * sizeof(crt_visibility), &fresh);
        if (rc != CRT_OK) return rc;
        if (fresh) CRT_CUDA(cudaMemsetAsync(ctx->halo_vis, 0xff, 2 * band_cap * sizeof(crt_visibility), ctx->stream));  // index -1: no hint yet
        // the kernels index records by the global pixel index: the band's first pixel, (H - b.y1) * W, lands on the slot's
        // first record (only the band's own pixels are read or written)
        const size_t first = (size_t)(H - b.y1) * W;
        crt_visibility* vis = (crt_visibility*)((uintptr_t)ctx->halo_vis + (uintptr_t)(k * band_cap) * sizeof(crt_visibility) -
                                                (uintptr_t)first * sizeof(crt_visibility));
        rc = raycast_rows(ctx, W, H, geom, raygen, b, vis, "halo_raycast");
        if (rc != CRT_OK) return rc;
        launchers(ctx).halo_surfaces(ctx->stream, tile_grid(W, b), W, H, b, tris60, vis, eye, g);
        rc = check_launch(ctx, "halo_surfaces");
        if (rc != CRT_OK) return rc;
    }
    ctx->halo_reach = h;
    ctx->halo_dims[0] = W;
    ctx->halo_dims[1] = H;
    return CRT_OK;
}
int which_of(const crt_restir_buffers* b, const crt_buffer& x) { return x.data == b->temporal.data ? 0 : x.data == b->reservoir0.data ? 1 : 2; }
// input and output of spatial pass k in fused mode
void pass_buffers(const crt_restir_buffers* b, int pass, crt_buffer* in, crt_buffer* out)
{
    if (pass == 0) { *in = b->temporal; *out = b->reservoir1; }
    else if (pass % 2) { *in = b->reservoir1; *out = b->reservoir0; }
    else { *in = b->reservoir0; *out = b->reservoir1; }
}
}  // namespace

extern "C" int crt_restir_output_buffer(crt_options options, const crt_restir_buffers* b, crt_buffer* out)
{
    CRT_REQUIRE(b && out, "null argument");
    const int passes = options.spatial_resampling_passes;
    if (fused(options) && (!options.use_spatial_resampling || passes <= 0)) *out = b->temporal;
    else *out = (passes % 2) ? b->reservoir1 : b->reservoir0;  // the reference's buf_output (10_restir_di.cpp:324-336)
    return CRT_OK;
}

extern "C" int crt_restir_is_fused(crt_options options) { return fused(options) ? 1 : 0; }

const char* const kNoSurfacesMsg = "unbiased reuse weights do not take a previous camera without the previous frame's surfaces: "
                                   "set it with crt_restir_set_previous_frame";

extern "C" int crt_restir_set_previous_camera(crt_ctx* ctx, const crt_raygen* previous_raygen)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_REQUIRE(!previous_raygen || ctx->reuse_mode != CRT_REUSE_UNBIASED, kNoSurfacesMsg);
    ctx->prev_cam_set = previous_raygen != nullptr;
    if (previous_raygen) ctx->prev_cam = *previous_raygen;
    ctx->prev_vis = crt_buffer{};
    if (!previous_raygen) ctx->prev_tris = crt_buffer{};
    return CRT_OK;
}

extern "C" int crt_restir_set_previous_frame(crt_ctx* ctx, const crt_raygen* previous_raygen, crt_buffer previous_visibility)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_REQUIRE(!previous_raygen || previous_visibility.data != nullptr, "null previous visibility buffer");
    ctx->prev_cam_set = previous_raygen != nullptr;
    if (previous_raygen) ctx->prev_cam = *previous_raygen;
    ctx->prev_vis = previous_raygen ? previous_visibility : crt_buffer{};
    if (!previous_raygen) ctx->prev_tris = crt_buffer{};
    return CRT_OK;
}

extern "C" int crt_restir_set_previous_triangles(crt_ctx* ctx, crt_buffer previous_triangles)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_REQUIRE(previous_triangles.data != nullptr || bsize(previous_triangles) == 0, "null previous triangle buffer");
    ctx->prev_tris = previous_triangles.data ? previous_triangles : crt_buffer{};
    return CRT_OK;
}

extern "C" int crt_restir_set_halo_surfaces(crt_ctx* ctx, int enable)
{
    CRT_REQUIRE(ctx, "null context");
    ctx->halo_surfaces = enable ? 1 : 0;
    return CRT_OK;
}

extern "C" int crt_restir_class_plane(crt_ctx* ctx, void** out)
{
    CRT_REQUIRE(ctx && out, "null argument");
    CRT_REQUIRE(ctx->gbuf, "no fused frame has run on this context yet");
    *out = (char*)ctx->gbuf + ctx->gbuf_pixels * 24;
    return CRT_OK;
}

extern "C" int crt_restir_frame_begin(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom, crt_buffer triangles,
                                      crt_raygen raygen, crt_float3 eye, crt_buffer lights, crt_options options,
                                      const crt_restir_buffers* b)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    int rc = check_buffers(W, H, b);
    if (rc != CRT_OK) return rc;
    const bool with_surfaces = ctx->prev_cam_set && ctx->prev_vis.data != nullptr;  // crt_restir_set_previous_frame
    if (with_surfaces)
    {
        CRT_CHECK_BUF(ctx->prev_vis, (size_t)W * H, "previous visibility");
        CRT_REQUIRE(ctx->prev_vis.data != b->visibility.data,
                    "the previous frame's Visibility must be a buffer of its own: this frame's raycast overwrites buffers->visibility");
    }
    const bool motion = ctx->prev_cam_set && ctx->prev_tris.data != nullptr;  // crt_restir_set_previous_triangles
    CRT_REQUIRE(!motion || bsize(ctx->prev_tris) == bsize(triangles),
                "the previous triangle array must hold as many triangles as the current one, in the same order");
    rc = raycast_or_prefetched(ctx, W, H, geom, triangles, raygen, b->visibility);
    if (rc != CRT_OK) return rc;
    ctx->frame_fused = fused(options);
    if (ctx->reuse_mode == CRT_REUSE_UNBIASED)
    {
        CRT_REQUIRE(!ctx->prev_cam_set || with_surfaces, kNoSurfacesMsg);
        CRT_REQUIRE(unbiased_rows_ok(ctx, H, options), kUnbiasedRowsMsg);
    }
    if (ctx->links_set)
    {
        // what the direct-store halo protocol (slab_p2p.cu) covers; anything else must use a host-side exchange
        CRT_REQUIRE(ctx->frame_fused, "slab links are set but these options take the per-kernel path: exchange AoS rows on the host");
        CRT_REQUIRE(!options.use_spatial_resampling || halo_rows_for(options.spatial_resampling_radius) <= kHaloRows,
                    "slab links mirror 87 halo rows: spatial_resampling_radius above 30 needs a host-side exchange");
        CRT_REQUIRE(!options.use_spatial_resampling || options.spatial_resampling_passes != 1,
                    "slab links need 0 or >= 2 spatial passes (one signal/wait per pass orders the neighbours)");
    }
    if (ctx->prev_cam_set)
    {
        // A look-up at another pixel reads rows this context may not compute (DESIGN.md section 11).  A host that renders a
        // row range gathers every slab's rows of `temporal` before this call (python/slabs.py: gather_history); the
        // direct-store links mirror the 87 halo rows only, so they cannot serve it.
        CRT_REQUIRE(!ctx->links_set, "temporal reprojection in the fused frame cannot run over the direct-store slab links: "
                                     "the host gathers the history rows (exchange mode)");
    }
    if (!fused(options))
    {
        rc = crt_generate_candidate(ctx, W, H, frame, geom, triangles, b->visibility, eye, lights, options, b->reservoir0);
        if (rc == CRT_OK)
            rc = motion              ? crt_temporal_resampling_reprojected_motion(ctx, W, H, frame, geom, triangles, b->visibility, eye,
                                                                                  options, ctx->prev_cam, ctx->prev_tris, ctx->prev_vis,
                                                                                  b->temporal, b->reservoir0)
                 : with_surfaces     ? crt_temporal_resampling_reprojected_surfaces(ctx, W, H, frame, geom, triangles, b->visibility, eye,
                                                                                    options, ctx->prev_cam, ctx->prev_vis, b->temporal,
                                                                                    b->reservoir0)
                 : ctx->prev_cam_set ? crt_temporal_resampling_reprojected(ctx, W, H, frame, geom, triangles, b->visibility, eye, options,
                                                                           ctx->prev_cam, b->temporal, b->reservoir0)
                                     : crt_temporal_resampling(ctx, W, H, frame, geom, triangles, b->visibility, eye, options, b->temporal, b->reservoir0);
        if (rc == CRT_OK) rc = crt_save_temporal_reservoir(ctx, W, H, b->reservoir0, b->temporal);
        return rc;
    }
    CRT_REQUIRE(triangles.data != nullptr, "null triangle buffer");
    CRT_REQUIRE(bsize(lights) == 0 || lights.data != nullptr, "null light buffer");
    CRT_REQUIRE(bsize(lights) < 0xffffffffull, "too many lights");
    const size_t n = (size_t)W * H;
    const Rows rows = rows_of(ctx, H);
    GBuf g;
    rc = ensure_gbuf(ctx, n, &g);
    if (rc != CRT_OK) return rc;
    ShadowQueue q{nullptr, nullptr, nullptr, 0};
    rc = queue_prepare(ctx, (size_t)(rows.y1 - rows.y0) * W, &q);
    if (rc != CRT_OK) return rc;
    const float* tris60 = (const float*)triangles.data;
    const crt_visibility* vis = (const crt_visibility*)b->visibility.data;
    const uint32_t n_lights = (uint32_t)bsize(lights);
    const SoaStore T = soa(b->temporal, n);
#if !defined(CRT_MUTATION_KEEP_TRACED)  // (a mutation build for tests/test_gpu_parity.py: the geometry test must then fail)
    if (geom->serial != ctx->history_serial || b->temporal.data != ctx->history_buffer)
    {
        // another geometry (or another history buffer) than last frame's: its traced marks are not ours to trust
        const size_t own_first = (size_t)(H - rows.y1) * W, own_n = (size_t)(rows.y1 - rows.y0) * W;
        if (own_n) k_clear_traced<<<sweep_blocks(ctx, own_n), 256, 0, ctx->stream>>>(own_first, own_n, T);
        rc = check_launch(ctx, "clear_traced");
        if (rc != CRT_OK) return rc;
        ctx->history_serial = geom->serial;
        ctx->history_buffer = b->temporal.data;
    }
#endif
    rc = halo_surfaces(ctx, W, H, geom, tris60, raygen, to_f3(eye), options, rows, g);
    if (rc != CRT_OK) return rc;
    const dim3 grid = tile_grid(W, rows);
    const bool exact = ctx->math_mode == CRT_MATH_EXACT;
    const HaloPeers peers = halo_peers(ctx, 0, rows, true, n);
    const LightRec* table = nullptr;
    uint32_t n_slots = n_lights;
    if (use_light_table(ctx))
    {
        rc = light_table_for(ctx, geom, tris60, (const uint32_t*)lights.data, n_lights, &table, &n_slots);
        if (rc != CRT_OK) return rc;
    }
    LightsTiles tiles{nullptr, (uint32_t)ctx->tiles_log2_t, (uint32_t)ctx->tiles_log2_s};
    if (light_tiles_on(ctx, n_lights))
    {
        rc = light_tiles_for(ctx, geom, table, n_slots, frame, &tiles.tiles);
        if (rc != CRT_OK) return rc;
    }
    Reprojection rp;
    const bool reproject = ctx->prev_cam_set && options.use_temporal_resampling;
    if (reproject)
    {
        // snapshot of last frame's history: this frame's records overwrite `temporal` while other pixels still look theirs up
        rc = grow(ctx->history_prev, ctx->history_prev_pixels, n, n * 72);
        if (rc != CRT_OK) return rc;
        CRT_CUDA(cudaMemcpyAsync(ctx->history_prev, b->temporal.data, n * 72, cudaMemcpyDeviceToDevice, ctx->stream));
        rp.history = SoaStore{(char*)ctx->history_prev, n};
        rp.prev_cam = ctx->prev_cam;
        rp.W = W;
        rp.H = H;
        rp.prev_vis = (const crt_visibility*)ctx->prev_vis.data;
        rp.prev_eye = to_f3(ctx->prev_cam.m_origin);
    }
    launchers(ctx).candidate_temporal(
        ctx->stream, exact, grid, W, H, rows, frame, geom->view(), tris60, vis, to_f3(eye), table,
        (const uint32_t*)lights.data, n_slots, options, T, g, q, peers, reproject ? &rp : nullptr, ctx->reuse_mode,
        tiles.tiles ? &tiles : nullptr, reproject && motion ? (const float*)ctx->prev_tris.data : nullptr);
    rc = check_launch(ctx, "candidate_temporal");
    if (rc != CRT_OK || !options.use_visibility_reuse) return rc;
    ShadowSink sink{nullptr, nullptr, 0, (uint32_t*)T.plane(0, 0)};
    if (peers.up) sink.up_plane0 = (uint32_t*)SoaStore{peers.up, n}.plane(0, 0);
    if (peers.down) sink.down_plane0 = (uint32_t*)SoaStore{peers.down, n}.plane(0, 0);
    sink.up_first_idx = (uint32_t)((size_t)(H - peers.up_end) * W);        // rows yi < up_end
    sink.down_end_idx = (uint32_t)((size_t)(H - peers.down_begin) * W);    // rows yi >= down_begin
    return queue_trace<kEpiSoaVisibility>(ctx, geom, q, sink);
}

extern "C" int crt_restir_spatial_pass(crt_ctx* ctx, int W, int H, int frame, int pass, crt_geometry geom,
                                       crt_buffer triangles, crt_float3 eye, crt_options options,
                                       const crt_restir_buffers* b)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    int rc = check_buffers(W, H, b);
    if (rc != CRT_OK) return rc;
    CRT_REQUIRE(pass >= 0, "negative pass index");
    if (!fused(options))
    {
        const bool odd = pass % 2;  // the reference's swap (10_restir_di.cpp:324-336): buf0 -> buf1, buf1 -> buf0, ...
        return crt_spatial_resampling(ctx, W, H, frame, pass, geom, triangles, b->visibility, eye, options,
                                      odd ? b->reservoir1 : b->reservoir0, odd ? b->reservoir0 : b->reservoir1);
    }
    if (!options.use_spatial_resampling) return CRT_OK;  // the reference's disabled pass is a copy
    CRT_REQUIRE(ctx->reuse_mode != CRT_REUSE_UNBIASED || unbiased_rows_ok(ctx, H, options), kUnbiasedRowsMsg);
    CRT_REQUIRE(ctx->reuse_mode != CRT_REUSE_UNBIASED || whole_image(ctx, H) ||
                    (ctx->halo_dims[0] == W && ctx->halo_dims[1] == H &&
                     halo_rows_for(options.spatial_resampling_radius) <= ctx->halo_reach),
                kHaloReachMsg);
    CRT_REQUIRE(ctx->gbuf && ctx->gbuf_pixels >= (size_t)W * H, "crt_restir_frame_begin has not run for this image size");
    const size_t n = (size_t)W * H;
    const Rows rows = rows_of(ctx, H);
    GBuf g;
    rc = ensure_gbuf(ctx, n, &g);
    if (rc != CRT_OK) return rc;
    crt_buffer in, out;
    pass_buffers(b, pass, &in, &out);
    // the last pass's output is only read by this rank's resolve: nothing to mirror
    const HaloPeers peers = pass + 1 < options.spatial_resampling_passes ? halo_peers(ctx, which_of(b, out), rows, false, n) : HaloPeers();
    launchers(ctx).spatial(
        ctx->stream, ctx->math_mode == CRT_MATH_EXACT, tile_grid(W, rows), W, H, rows, frame, pass, geom->view(), to_f3(eye),
        options, soa(in, n), soa(out, n), g, peers, ctx->reuse_mode);
    return check_launch(ctx, "spatial_fast");
}

extern "C" int crt_restir_frame_end(crt_ctx* ctx, int W, int H, crt_geometry geom, crt_buffer triangles, crt_float3 eye,
                                    crt_options options, const crt_restir_buffers* b)
{
    CRT_REQUIRE(ctx && geom, "null context or geometry");
    int rc = check_buffers(W, H, b);
    if (rc != CRT_OK) return rc;
    CRT_JOIN_TAIL(ctx);  // the previous frame's tail owns the accumulation / pixel buffers and the second ray queue until here
    crt_buffer fin;
    crt_restir_output_buffer(options, b, &fin);
    if (!fused(options))
    {
        rc = crt_resolve(ctx, b->accumulation, W, H, geom, triangles, b->visibility, eye, options, fin);
        if (rc == CRT_OK) rc = crt_tone_mapping(ctx, b->pixels, b->accumulation, W, H);
        return rc;
    }
    CRT_REQUIRE(triangles.data != nullptr, "null triangle buffer");
    CRT_REQUIRE(ctx->gbuf && ctx->gbuf_pixels >= (size_t)W * H, "crt_restir_frame_begin has not run for this image size");
    const size_t n = (size_t)W * H;
    const Rows rows = rows_of(ctx, H);
    GBuf g;
    rc = ensure_gbuf(ctx, n, &g);
    if (rc != CRT_OK) return rc;
    const bool overlap = ctx->overlap != 0 && !ctx->profiling;
    ShadowQueue q{nullptr, nullptr, nullptr, 0};
    rc = queue_prepare(ctx, (size_t)(rows.y1 - rows.y0) * W, &q, overlap ? 1 : 0);
    if (rc != CRT_OK) return rc;
    crt_float4* accum = (crt_float4*)b->accumulation.data;
    launchers(ctx).resolve(
        ctx->stream, tile_grid(W, rows), accum, W, H, rows, (const float*)triangles.data,
        (const crt_visibility*)b->visibility.data, soa(fin, n), g, q, options.accumulate,
        ctx->resolve_reuse && options.use_visibility_reuse);
    rc = check_launch(ctx, "resolve_fast");
    if (rc != CRT_OK) return rc;
    if (!overlap)
    {
        rc = queue_trace<kEpiResolve>(ctx, geom, q, ShadowSink{nullptr, accum, options.accumulate, nullptr});
        if (rc != CRT_OK) return rc;
        return crt_tone_mapping(ctx, b->pixels, b->accumulation, W, H);
    }
    // The tail — resolve rays, then tone mapping — goes to the second stream: it reads only its own ray queue (shading
    // factors included) and reads / writes accumulation and pixels, none of which the next frame touches before its own
    // crt_restir_frame_end, and that call (like every other entry point that touches those buffers) orders itself after
    // this tail first (join_tail at the top of this function).
    CRT_CUDA(cudaEventRecord(ctx->ev_head, ctx->stream));
    CRT_CUDA(cudaStreamWaitEvent(ctx->tail_stream, ctx->ev_head, 0));
    rc = queue_trace<kEpiResolve>(ctx, geom, q, ShadowSink{nullptr, accum, options.accumulate, nullptr}, ctx->tail_stream);
    if (rc != CRT_OK) return rc;
    rc = tone_mapping_on(ctx, ctx->tail_stream, b->pixels, b->accumulation, W, H);
    if (rc != CRT_OK) return rc;
    CRT_CUDA(cudaEventRecord(ctx->ev_tail, ctx->tail_stream));
    ctx->tail_pending = true;
    return CRT_OK;
}

extern "C" int crt_restir_di_frame(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom, crt_buffer triangles,
                                   crt_raygen raygen, crt_float3 eye, crt_buffer lights, crt_options options,
                                   const crt_restir_buffers* b)
{
    int rc = crt_restir_frame_begin(ctx, W, H, frame, geom, triangles, raygen, eye, lights, options, b);
    for (int pass = 0; rc == CRT_OK && pass < options.spatial_resampling_passes; pass++)
        rc = crt_restir_spatial_pass(ctx, W, H, frame, pass, geom, triangles, eye, options, b);
    if (rc == CRT_OK) rc = crt_restir_frame_end(ctx, W, H, geom, triangles, eye, options, b);
    return rc;
}

extern "C" int crt_reservoir_export_aos(crt_ctx* ctx, int W, int H, crt_buffer soa_storage, crt_buffer aos_out)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_CHECK_IMAGE(W, H);
    const size_t n = (size_t)W * H;
    CRT_CHECK_BUF(soa_storage, n, "SoA reservoir");
    CRT_CHECK_BUF(aos_out, n, "AoS reservoir");
    CRT_REQUIRE(soa_storage.data != aos_out.data, "conversion cannot run in place");
    k_soa_to_aos<<<sweep_blocks(ctx, n), 256, 0, ctx->stream>>>(n, soa(soa_storage, n), (crt_reservoir*)aos_out.data);
    return check_launch(ctx, "soa_to_aos");
}

extern "C" int crt_reservoir_import_aos(crt_ctx* ctx, int W, int H, crt_buffer aos_in, crt_buffer soa_storage)
{
    CRT_REQUIRE(ctx, "null context");
    CRT_CHECK_IMAGE(W, H);
    const size_t n = (size_t)W * H;
    CRT_CHECK_BUF(soa_storage, n, "SoA reservoir");
    CRT_CHECK_BUF(aos_in, n, "AoS reservoir");
    CRT_REQUIRE(soa_storage.data != aos_in.data, "conversion cannot run in place");
    k_aos_to_soa<<<sweep_blocks(ctx, n), 256, 0, ctx->stream>>>(n, (const crt_reservoir*)aos_in.data, soa(soa_storage, n));
    return check_launch(ctx, "aos_to_soa");
}
#endif  // !CRT_AUX_TU
