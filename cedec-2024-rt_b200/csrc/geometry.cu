// geometry.cu — crt_build_geometry / crt_destroy_geometry / ray probes.
// Replaces hiprtCreateContext + buildHiprtGeometry (10_restir_di.cpp:74-79,220; common/loader.hpp:68-112):
// the BVH is built on the GPU from the device-resident reference Triangle array, synchronously.
#include <atomic>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <stdarg.h>
#include <stdlib.h>

#include "bvh_build.cuh"
#include "ctx.cuh"
#include "restir_core.cuh"

namespace crt
{
static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}
const char* last_error() { return g_err; }

constexpr int kBuildBlock = 256;

__global__ void __launch_bounds__(kBuildBlock) k_init_bounds(uint32_t* bounds6)
{
    if (threadIdx.x < 3) bounds6[threadIdx.x] = 0xffffffffu;
    else if (threadIdx.x < 6) bounds6[threadIdx.x] = 0u;
}
__global__ void __launch_bounds__(kBuildBlock) k_tri_bounds(uint32_t n, const float* tris60, uint32_t* bounds6)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) tri_bounds(i, tris60, bounds6);
}
__global__ void __launch_bounds__(kBuildBlock)
    k_morton(uint32_t n, const float* tris60, f3 lo, f3 inv_extent, uint64_t* keys, uint32_t* idx)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = morton_key(i, tris60, lo, inv_extent);
    idx[i] = i;
}
__global__ void __launch_bounds__(kBuildBlock) k_lbvh_node(uint32_t n_inner, const uint64_t* keys, BinTree bt)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_inner) lbvh_node(i, keys, bt);
}
__global__ void __launch_bounds__(kBuildBlock)
    k_lbvh_refit(uint32_t n, const float* tris60, const uint32_t* sorted_idx, float pad, BinTree bt)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) lbvh_refit(i, tris60, sorted_idx, pad, bt);
}
__global__ void __launch_bounds__(kBuildBlock)
    k_ploc_init(uint32_t n, const float* tris60, const uint32_t* sorted_idx, float pad, BinTree bt, uint32_t* node_out,
                float* box_out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) ploc_init_leaf(i, tris60, sorted_idx, pad, bt, node_out, box_out);
}
__global__ void __launch_bounds__(kBuildBlock) k_ploc_nn(PlocRound p)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < p.m) ploc_nn(i, p);
}
__global__ void __launch_bounds__(kBuildBlock) k_ploc_flag(PlocRound p)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < p.m) ploc_flag(i, p);
}
// also leaves the round's totals (survivors | merges << 32) in *total for the host
__global__ void __launch_bounds__(kBuildBlock)
    k_ploc_apply(PlocRound p, const unsigned long long* scan, uint32_t id_top, BinTree bt, unsigned long long* total)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.m) return;
    ploc_apply(i, p, scan, id_top, bt);
    if (i == p.m - 1) *total = scan[i] + p.flag[i];
}
__global__ void __launch_bounds__(kBuildBlock)
    k_collapse(uint32_t n_items, const CollapseItem* items, const float* tris60, const uint32_t* sorted_idx,
               BinTree bt, WideOut out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_items) collapse_item(items[i], tris60, sorted_idx, bt, out);
}

// RAII for the build's temporaries
struct DevMem
{
    void* p = nullptr;
    ~DevMem()
    {
        if (p) cudaFree(p);
    }
    template <class T>
    T* as()
    {
        return (T*)p;
    }
};
#define CRT_ALLOC(mem, bytes) CRT_CUDA(cudaMalloc(&(mem).p, (bytes) ? (bytes) : 16))

static int build(crt_ctx* ctx, const crt_triangle* d_tris, size_t n_sz, crt_geometry_t* g)
{
    cudaStream_t st = ctx->stream;
    const uint32_t n = (uint32_t)n_sz;
    const float* tris60 = (const float*)d_tris;
    g->src = d_tris;
    g->n_tris = n;
    g->device = ctx->device;
    if (const char* e = getenv("CRT_POSTPONE")) g->postpone_ratio = (float)atof(e);

    if (n == 0)
    {
        WideNode root;
        memset(&root, 0, sizeof root);
        for (int s = 0; s < 8; s++)
            for (int a = 0; a < 3; a++) root.qlo[a][s] = 255;
        root.ex = root.ey = root.ez = 127;
        CRT_CUDA(cudaMalloc((void**)&g->nodes, sizeof(WideNode)));
        CRT_CUDA(cudaMalloc((void**)&g->tris, sizeof(WideTri)));
        CRT_CUDA(cudaMemcpyAsync(g->nodes, &root, sizeof root, cudaMemcpyHostToDevice, st));
        CRT_CUDA(cudaStreamSynchronize(st));
        g->n_nodes = 1;
        g->max_depth = 1;
        return CRT_OK;
    }

    cudaEvent_t e0, e1;
    CRT_CUDA(cudaEventCreate(&e0));
    CRT_CUDA(cudaEventCreate(&e1));
    CRT_CUDA(cudaEventRecord(e0, st));

    // ---- 1: scene bounds
    DevMem m_bounds;
    CRT_ALLOC(m_bounds, 6 * sizeof(uint32_t));
    k_init_bounds<<<1, kBuildBlock, 0, st>>>(m_bounds.as<uint32_t>());
    k_tri_bounds<<<div_up(n, kBuildBlock), kBuildBlock, 0, st>>>(n, tris60, m_bounds.as<uint32_t>());
    uint32_t hb[6];
    CRT_CUDA(cudaMemcpyAsync(hb, m_bounds.p, sizeof hb, cudaMemcpyDeviceToHost, st));
    CRT_CUDA(cudaStreamSynchronize(st));
    float lo[3], hi[3], max_abs = 0.0f;
    for (int a = 0; a < 3; a++)
    {
        lo[a] = ordered_to_float(hb[a]);
        hi[a] = ordered_to_float(hb[3 + a]);
        max_abs = fmaxf(max_abs, fmaxf(fabsf(lo[a]), fabsf(hi[a])));
    }
    // pad >= rounding error of the reference triangle test and of the slab arithmetic:
    // 64 ulp(1) x the largest coordinate magnitude (DESIGN.md, "conservative culling")
    float pad_scale = 64.0f;
    if (const char* s = getenv("CRT_BVH_PAD_ULPS")) pad_scale = (float)atof(s);
    g->pad = pad_scale * 5.9604645e-8f * fmaxf(max_abs, 1.0f);
    f3 inv_extent;
    inv_extent.x = hi[0] > lo[0] ? 1.0f / (hi[0] - lo[0]) : 0.0f;
    inv_extent.y = hi[1] > lo[1] ? 1.0f / (hi[1] - lo[1]) : 0.0f;
    inv_extent.z = hi[2] > lo[2] ? 1.0f / (hi[2] - lo[2]) : 0.0f;

    // ---- 2: Morton keys + radix sort
    DevMem m_keys, m_keys2, m_idx, m_idx2, m_sort;
    CRT_ALLOC(m_keys, n * sizeof(uint64_t));
    CRT_ALLOC(m_keys2, n * sizeof(uint64_t));
    CRT_ALLOC(m_idx, n * sizeof(uint32_t));
    CRT_ALLOC(m_idx2, n * sizeof(uint32_t));
    k_morton<<<div_up(n, kBuildBlock), kBuildBlock, 0, st>>>(n, tris60, f3{lo[0], lo[1], lo[2]}, inv_extent,
                                                            m_keys.as<uint64_t>(), m_idx.as<uint32_t>());
    size_t sort_bytes = 0;
    CRT_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, m_keys.as<uint64_t>(), m_keys2.as<uint64_t>(),
                                             m_idx.as<uint32_t>(), m_idx2.as<uint32_t>(), (int)n, 0, 63, st));
    CRT_ALLOC(m_sort, sort_bytes);
    CRT_CUDA(cub::DeviceRadixSort::SortPairs(m_sort.p, sort_bytes, m_keys.as<uint64_t>(), m_keys2.as<uint64_t>(),
                                             m_idx.as<uint32_t>(), m_idx2.as<uint32_t>(), (int)n, 0, 63, st));
    const uint64_t* keys = m_keys2.as<uint64_t>();
    const uint32_t* sorted_idx = m_idx2.as<uint32_t>();

    // ---- 3/4: binary radix tree + bottom-up boxes
    const uint32_t n_inner = n - 1;
    DevMem m_left, m_right, m_parent, m_first, m_count, m_box, m_visits, m_cost, m_split;
    CRT_ALLOC(m_left, n_inner * sizeof(uint32_t));
    CRT_ALLOC(m_right, n_inner * sizeof(uint32_t));
    CRT_ALLOC(m_parent, (2 * (size_t)n - 1) * sizeof(uint32_t));
    CRT_ALLOC(m_first, n_inner * sizeof(uint32_t));
    CRT_ALLOC(m_count, n_inner * sizeof(uint32_t));
    CRT_ALLOC(m_box, (2 * (size_t)n - 1) * 6 * sizeof(float));
    CRT_ALLOC(m_visits, n_inner * sizeof(uint32_t));
    CRT_ALLOC(m_cost, (2 * (size_t)n - 1) * 7 * sizeof(float));
    CRT_ALLOC(m_split, (2 * (size_t)n - 1) * 8);
    CRT_CUDA(cudaMemsetAsync(m_visits.p, 0, n_inner ? n_inner * sizeof(uint32_t) : 16, st));
    BinTree bt;
    bt.n = n;
    bt.left = m_left.as<uint32_t>();
    bt.right = m_right.as<uint32_t>();
    bt.parent = m_parent.as<uint32_t>();
    bt.first = m_first.as<uint32_t>();
    bt.count = m_count.as<uint32_t>();
    bt.box = m_box.as<float>();
    bt.visits = m_visits.as<uint32_t>();
    bt.cost = m_cost.as<float>();
    bt.split = m_split.as<uint8_t>();
    const char* builder = getenv("CRT_BVH_BUILDER");
    int ploc_rounds = 0;
    if (builder && !strcmp(builder, "lbvh"))
    {
        if (n_inner) k_lbvh_node<<<div_up(n_inner, kBuildBlock), kBuildBlock, 0, st>>>(n_inner, keys, bt);
        k_lbvh_refit<<<div_up(n, kBuildBlock), kBuildBlock, 0, st>>>(n, tris60, sorted_idx, g->pad, bt);
    }
    else
    {
        // PLOC rounds: nearest neighbour, flag, scan, apply; the host reads the survivor count after each round
        DevMem m_na, m_nb, m_ba, m_bb, m_nn, m_flag, m_scan, m_total, m_scan_tmp;
        CRT_ALLOC(m_na, n * sizeof(uint32_t));
        CRT_ALLOC(m_nb, n * sizeof(uint32_t));
        CRT_ALLOC(m_ba, (size_t)n * 8 * sizeof(float));
        CRT_ALLOC(m_bb, (size_t)n * 8 * sizeof(float));
        CRT_ALLOC(m_nn, n * sizeof(uint32_t));
        CRT_ALLOC(m_flag, n * sizeof(unsigned long long));
        CRT_ALLOC(m_scan, n * sizeof(unsigned long long));
        CRT_ALLOC(m_total, sizeof(unsigned long long));
        size_t scan_bytes = 0;
        CRT_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, m_flag.as<unsigned long long>(),
                                               m_scan.as<unsigned long long>(), (int)n, st));
        CRT_ALLOC(m_scan_tmp, scan_bytes);
        uint32_t* node_in = m_na.as<uint32_t>();
        uint32_t* node_out = m_nb.as<uint32_t>();
        float* box_in = m_ba.as<float>();
        float* box_out = m_bb.as<float>();
        k_ploc_init<<<div_up(n, kBuildBlock), kBuildBlock, 0, st>>>(n, tris60, sorted_idx, g->pad, bt, node_in, box_in);
        uint32_t m = n, id_top = n >= 2 ? n - 2 : 0;
        while (m > 1)
        {
            PlocRound pr{m, node_in, box_in, m_nn.as<uint32_t>(), m_flag.as<unsigned long long>(), node_out, box_out};
            const unsigned blocks = div_up(m, kBuildBlock);
            k_ploc_nn<<<blocks, kBuildBlock, 0, st>>>(pr);
            k_ploc_flag<<<blocks, kBuildBlock, 0, st>>>(pr);
            CRT_CUDA(cub::DeviceScan::ExclusiveSum(m_scan_tmp.p, scan_bytes, m_flag.as<unsigned long long>(),
                                                   m_scan.as<unsigned long long>(), (int)m, st));
            k_ploc_apply<<<blocks, kBuildBlock, 0, st>>>(pr, m_scan.as<unsigned long long>(), id_top, bt,
                                                        m_total.as<unsigned long long>());
            unsigned long long total = 0;
            CRT_CUDA(cudaMemcpyAsync(&total, m_total.p, sizeof total, cudaMemcpyDeviceToHost, st));
            CRT_CUDA(cudaStreamSynchronize(st));
            const uint32_t merges = (uint32_t)(total >> 32), survivors = (uint32_t)(total & 0xffffffffull);
            if (merges == 0 || survivors >= m)
            {
                set_error("PLOC round made no progress (%u clusters)", m);
                return CRT_ECUDA;
            }
            id_top -= merges;
            m = survivors;
            uint32_t* tn = node_in; node_in = node_out; node_out = tn;
            float* tb = box_in; box_in = box_out; box_out = tb;
            ++ploc_rounds;
        }
        ctx->launches += 1 + 4 * (unsigned long long)ploc_rounds;
    }

    // ---- 5: collapse, one launch per level of the wide tree
    DevMem m_nodes, m_q0, m_q1, m_counters;
    const size_t node_cap = (size_t)n + 1;
    CRT_ALLOC(m_nodes, node_cap * sizeof(WideNode));
    CRT_CUDA(cudaMalloc((void**)&g->tris, (size_t)n * sizeof(WideTri)));
    CRT_ALLOC(m_q0, node_cap * sizeof(CollapseItem));
    CRT_ALLOC(m_q1, node_cap * sizeof(CollapseItem));
    CRT_ALLOC(m_counters, 4 * sizeof(uint32_t));  // node_count, tri_count, next_count
    const uint32_t init_counters[4] = {1u, 0u, 0u, 0u};
    CRT_CUDA(cudaMemcpyAsync(m_counters.p, init_counters, sizeof init_counters, cudaMemcpyHostToDevice, st));
    const CollapseItem root_item{0u, 0u};
    CRT_CUDA(cudaMemcpyAsync(m_q0.p, &root_item, sizeof root_item, cudaMemcpyHostToDevice, st));
    WideOut out;
    out.nodes = m_nodes.as<WideNode>();
    out.tris = g->tris;
    out.node_count = m_counters.as<uint32_t>() + 0;
    out.tri_count = m_counters.as<uint32_t>() + 1;
    out.next_count = m_counters.as<uint32_t>() + 2;
    CollapseItem* q_in = m_q0.as<CollapseItem>();
    CollapseItem* q_out = m_q1.as<CollapseItem>();
    uint32_t n_items = 1;
    int depth = 0;
    g->level_begin.assign(1, 0u);
    while (n_items)
    {
        depth++;
        g->level_begin.push_back(g->level_begin.back() + n_items);  // this level's nodes end where the next level's begin
        out.next = q_out;
        CRT_CUDA(cudaMemsetAsync(out.next_count, 0, sizeof(uint32_t), st));
        k_collapse<<<div_up(n_items, kBuildBlock), kBuildBlock, 0, st>>>(n_items, q_in, tris60, sorted_idx, bt, out);
        CRT_CUDA(cudaMemcpyAsync(&n_items, out.next_count, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        CRT_CUDA(cudaStreamSynchronize(st));
        CollapseItem* t = q_in;
        q_in = q_out;
        q_out = t;
        if (depth > 4096)
        {
            set_error("BVH collapse did not terminate");
            return CRT_ECUDA;
        }
    }
    uint32_t counters[4];
    CRT_CUDA(cudaMemcpyAsync(counters, m_counters.p, sizeof counters, cudaMemcpyDeviceToHost, st));
    CRT_CUDA(cudaStreamSynchronize(st));
    if (counters[1] != n)
    {
        set_error("BVH build wrote %u triangle records for %u triangles", counters[1], n);
        return CRT_ECUDA;
    }
    g->n_nodes = counters[0];
    g->max_depth = depth;
    CRT_CUDA(cudaMalloc((void**)&g->nodes, g->n_nodes * sizeof(WideNode)));
    CRT_CUDA(cudaMemcpyAsync(g->nodes, m_nodes.p, g->n_nodes * sizeof(WideNode), cudaMemcpyDeviceToDevice, st));
    CRT_CUDA(cudaEventRecord(e1, st));
    CRT_CUDA(cudaStreamSynchronize(st));
    CRT_CUDA(cudaEventElapsedTime(&g->build_ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CRT_CUDA(cudaGetLastError());
    ctx->launches += 5 + depth;
    if (2 * depth > kStackSize)
    {
        set_error("wide BVH depth %d exceeds the traversal stack (%d entries, two per level)", depth, kStackSize);
        return CRT_ESTACK;
    }
    return CRT_OK;
}

// ---- refit
__global__ void __launch_bounds__(kBuildBlock) k_refit_tris(uint32_t n, const float* tris60, WideTri* tris)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) refit_tri(i, tris60, tris);
}
__global__ void __launch_bounds__(kBuildBlock)
    k_refit_nodes(uint32_t first, uint32_t count, WideNode* nodes, const WideTri* tris, float* node_box, float pad)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) refit_node(first + i, nodes, tris, node_box, pad);
}
static std::atomic<unsigned long long> g_next_serial{1};

static int refit(crt_ctx* ctx, crt_geometry_t* g)
{
    cudaStream_t st = ctx->stream;
    const uint32_t n = (uint32_t)g->n_tris;
    if (n == 0) return CRT_OK;
    const float* tris60 = (const float*)g->src;
    cudaEvent_t e0, e1;
    CRT_CUDA(cudaEventCreate(&e0));
    CRT_CUDA(cudaEventCreate(&e1));
    CRT_CUDA(cudaEventRecord(e0, st));
    // the padding follows the largest coordinate (build(), step 1)
    DevMem m_bounds;
    CRT_ALLOC(m_bounds, 6 * sizeof(uint32_t));
    k_init_bounds<<<1, kBuildBlock, 0, st>>>(m_bounds.as<uint32_t>());
    k_tri_bounds<<<div_up(n, kBuildBlock), kBuildBlock, 0, st>>>(n, tris60, m_bounds.as<uint32_t>());
    uint32_t hb[6];
    CRT_CUDA(cudaMemcpyAsync(hb, m_bounds.p, sizeof hb, cudaMemcpyDeviceToHost, st));
    CRT_CUDA(cudaStreamSynchronize(st));
    float max_abs = 0.0f;
    for (int a = 0; a < 6; a++) max_abs = fmaxf(max_abs, fabsf(ordered_to_float(hb[a])));
    float pad_scale = 64.0f;
    if (const char* s = getenv("CRT_BVH_PAD_ULPS")) pad_scale = (float)atof(s);
    g->pad = pad_scale * 5.9604645e-8f * fmaxf(max_abs, 1.0f);
    if (!g->node_box) CRT_CUDA(cudaMalloc((void**)&g->node_box, g->n_nodes * 6 * sizeof(float)));
    k_refit_tris<<<div_up(n, kBuildBlock), kBuildBlock, 0, st>>>(n, tris60, g->tris);
    const int levels = (int)g->level_begin.size() - 1;
    for (int l = levels - 1; l >= 0; l--)
    {
        const uint32_t first = g->level_begin[l], count = g->level_begin[l + 1] - first;
        if (count) k_refit_nodes<<<div_up(count, kBuildBlock), kBuildBlock, 0, st>>>(first, count, g->nodes, g->tris, g->node_box, g->pad);
    }
    CRT_CUDA(cudaEventRecord(e1, st));
    CRT_CUDA(cudaStreamSynchronize(st));
    CRT_CUDA(cudaEventElapsedTime(&g->refit_ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CRT_CUDA(cudaGetLastError());
    ctx->launches += 3 + levels;
    g->serial = g_next_serial.fetch_add(1);  // visibility traced against the old positions is history (kernels_fast.cu)
    g->light_table_key = nullptr;            // emissive triangles may have moved: the light records are rebuilt on use
    return CRT_OK;
}

// ---- ray probes
template <bool ANY>
__global__ void __launch_bounds__(256) k_trace(Bvh bvh, size_t n, const float* org, const float* dir, float tmin,
                                               float tmax, int32_t* out_prim, float* out_tuv)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Hit h;
    const bool hit = trace<ANY>(bvh, f3{org[3 * i], org[3 * i + 1], org[3 * i + 2]},
                                f3{dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]}, tmin, tmax, h);
    if (ANY) out_prim[i] = hit ? 1 : 0;
    else
    {
        out_prim[i] = h.prim;
        out_tuv[3 * i + 0] = h.prim < 0 ? 0.0f : h.t;
        out_tuv[3 * i + 1] = h.u;
        out_tuv[3 * i + 2] = h.v;
    }
}

// exhaustive search, warp per ray: lanes stride over the triangles, then the warp reduces with the
// same rule (smaller t, then larger primitive id)
__global__ void __launch_bounds__(256) k_trace_brute(const float* tris60, uint32_t n_tris, size_t n, const float* org,
                                                     const float* dir, float tmin, float tmax, int32_t* out_prim,
                                                     float* out_tuv)
{
    const size_t ray = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (ray >= n) return;
    const f3 ro{org[3 * ray], org[3 * ray + 1], org[3 * ray + 2]}, rd{dir[3 * ray], dir[3 * ray + 1], dir[3 * ray + 2]};
    float bt = tmax, bu = 0.0f, bv = 0.0f;
    int bp = -1;
    for (uint32_t i = lane; i < n_tris; i += 32)
    {
        const BuildTri t = load_build_tri(tris60, i);
        float tt, u, v;
        if (ray_triangle(ro, rd, tmin, bt, t.v0, t.v1, t.v2, tt, u, v))
        {
            // within a lane indices ascend, so an accepted t <= bt always replaces (04_ao.cu:14-24)
            bt = tt; bu = u; bv = v; bp = (int)i;
        }
    }
    for (int off = 16; off; off >>= 1)
    {
        const float ot = __shfl_down_sync(0xffffffffu, bt, off), ou = __shfl_down_sync(0xffffffffu, bu, off),
                    ov = __shfl_down_sync(0xffffffffu, bv, off);
        const int op = __shfl_down_sync(0xffffffffu, bp, off);
        if (op >= 0 && (bp < 0 || ot < bt || (ot == bt && op > bp)))
        {
            bt = ot; bu = ou; bv = ov; bp = op;
        }
    }
    if (lane == 0)
    {
        out_prim[ray] = bp;
        out_tuv[3 * ray + 0] = bp < 0 ? 0.0f : bt;
        out_tuv[3 * ray + 1] = bu;
        out_tuv[3 * ray + 2] = bv;
    }
}

// ---- the slot table of power-proportional light selection (restir_core.cuh: light_power .. slot_owner).  Rebuilt per
// (geometry, light list, K) and after every refit or crt_lights_changed, so a host that animates emitters pays it per frame.
__global__ void __launch_bounds__(kBuildBlock)
    k_light_power(uint32_t n, const float* tris60, const uint32_t* lights, float* power, uint32_t* pmax_bits)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const float p = i < n ? light_power(tris60, CRT_LDG(lights + i)) : 0.0f;
    if (i < n) power[i] = p;
    // non-negative finite floats order like their bit patterns: the maximum is independent of the order of the atomics
    const uint32_t m = __reduce_max_sync(0xffffffffu, __float_as_uint(p));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(pmax_bits, m);
}
__global__ void __launch_bounds__(kBuildBlock)
    k_light_quantise(uint32_t n, const float* power, const uint32_t* pmax_bits, unsigned long long* q)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) q[i] = light_quantum(power[i], __uint_as_float(*pmax_bits));
    else if (i == n) q[n] = 0ull;  // the exclusive scan's last element is then S = S_n
}
__global__ void __launch_bounds__(kBuildBlock)
    k_light_starts(uint32_t n, uint32_t K, const unsigned long long* prefix, uint32_t* start)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) start[i] = light_start(i, n, K, prefix[i], prefix[n]);
    else if (i == n) start[n] = K;
}
// one thread per slot: a binary search over the starts keeps the work even when one light owns most of the slots
__global__ void __launch_bounds__(kBuildBlock)
    k_light_slots(uint32_t K, uint32_t n, const uint32_t* start, const float* tris60, const uint32_t* lights, LightRec* table)
{
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < K; s += gridDim.x * blockDim.x)
    {
        const uint32_t i = slot_owner(start, n, s);
        table[s] = light_rec(tris60, CRT_LDG(lights + i), slot_sel(CRT_LDG(start + i + 1) - CRT_LDG(start + i), K));
    }
}
int build_light_slots(crt_ctx* ctx, crt_geometry geom, const float* tris60, const uint32_t* lights, uint32_t n, int log2_slots,
                      LightRec* table)
{
    const uint32_t K = 1u << log2_slots;
    cudaStream_t st = ctx->stream;
    size_t scan_bytes = 0;
    CRT_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                           (int)n + 1, st));
    // scratch: q and its prefix (n + 1 each), power (n), starts (n + 1), the maximum, CUB's temporary storage
    const size_t q_bytes = ((size_t)n + 1) * 8, off_prefix = q_bytes, off_power = 2 * q_bytes,
                 off_start = off_power + (((size_t)n * 4 + 255) & ~(size_t)255), off_max = off_start + ((((size_t)n + 1) * 4 + 255) & ~(size_t)255),
                 off_tmp = off_max + 256, bytes = off_tmp + scan_bytes;
    int rc = grow(geom->light_scratch, geom->light_scratch_bytes, bytes, bytes);
    if (rc != CRT_OK) return rc;
    char* base = (char*)geom->light_scratch;
    unsigned long long *q = (unsigned long long*)base, *prefix = (unsigned long long*)(base + off_prefix);
    float* power = (float*)(base + off_power);
    uint32_t *start = (uint32_t*)(base + off_start), *pmax = (uint32_t*)(base + off_max);
    CRT_CUDA(cudaMemsetAsync(pmax, 0, 4, st));
    k_light_power<<<div_up(n, kBuildBlock), kBuildBlock, 0, st>>>(n, tris60, lights, power, pmax);
    rc = check_launch(ctx, "light_power");
    if (rc != CRT_OK) return rc;
    k_light_quantise<<<div_up((size_t)n + 1, kBuildBlock), kBuildBlock, 0, st>>>(n, power, pmax, q);
    rc = check_launch(ctx, "light_quantise");
    if (rc != CRT_OK) return rc;
    CRT_CUDA(cub::DeviceScan::ExclusiveSum(base + off_tmp, scan_bytes, q, prefix, (int)n + 1, st));
    rc = check_launch(ctx, "light_scan");
    if (rc != CRT_OK) return rc;
    k_light_starts<<<div_up((size_t)n + 1, kBuildBlock), kBuildBlock, 0, st>>>(n, K, prefix, start);
    rc = check_launch(ctx, "light_starts");
    if (rc != CRT_OK) return rc;
    const size_t want = div_up(K, kBuildBlock), cap = (size_t)ctx->sm_count * 16;
    k_light_slots<<<(unsigned)(want < cap ? want : cap), kBuildBlock, 0, st>>>(K, n, start, tris60, lights, table);
    return check_launch(ctx, "light_slots");
}

// ---- presampled light tiles (restir_core.cuh: light_tile_slot): one thread per entry, a pure function of its index
__global__ void __launch_bounds__(kBuildBlock)
    k_light_tiles(const LightRec* src, uint32_t K, uint32_t frame, uint32_t log2_s, uint32_t count, LightRec* tiles)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) tiles[i] = src[light_tile_slot(frame, i >> log2_s, i & ((1u << log2_s) - 1u), K)];
}
int build_light_tiles(crt_ctx* ctx, const LightRec* src, uint32_t K, int frame, int log2_t, int log2_s, LightRec* tiles)
{
    const uint32_t count = 1u << (log2_t + log2_s);
    k_light_tiles<<<div_up(count, kBuildBlock), kBuildBlock, 0, ctx->stream>>>(src, K, (uint32_t)frame, (uint32_t)log2_s, count, tiles);
    return check_launch(ctx, "light_tiles");
}
}  // namespace crt

using namespace crt;

extern "C" const char* crt_last_error(void) { return crt::last_error(); }

extern "C" int crt_build_geometry(crt_ctx* ctx, const crt_triangle* d_triangles, size_t n, crt_geometry* out)
{
    CRT_REQUIRE(ctx && out, "null argument");
    CRT_REQUIRE(n == 0 || d_triangles, "null triangle array");
    CRT_REQUIRE(n < 0x7fffffffull, "too many triangles");
    CRT_CUDA(cudaSetDevice(ctx->device));
    crt_geometry_t* g = new crt_geometry_t;
    g->serial = g_next_serial.fetch_add(1);
    const int rc = build(ctx, d_triangles, n, g);
    if (rc != CRT_OK)
    {
        if (g->nodes) cudaFree(g->nodes);
        if (g->tris) cudaFree(g->tris);
        delete g;
        *out = nullptr;
        return rc;
    }
    *out = g;
    return CRT_OK;
}

extern "C" int crt_refit_geometry(crt_ctx* ctx, crt_geometry g)
{
    CRT_REQUIRE(ctx && g, "null context or geometry");
    CRT_REQUIRE(g->device == ctx->device, "geometry belongs to another device");
    CRT_CUDA(cudaSetDevice(ctx->device));
    return refit(ctx, g);
}

extern "C" int crt_lights_changed(crt_ctx* ctx, crt_geometry g)
{
    CRT_REQUIRE(ctx && g, "null context or geometry");
    g->light_table_key = nullptr;  // the records (and in power mode the slot counts) are rebuilt at the next use
    return CRT_OK;
}

extern "C" int crt_destroy_geometry(crt_ctx* ctx, crt_geometry g)
{
    CRT_REQUIRE(ctx, "null context");
    if (!g) return CRT_OK;
    CRT_CUDA(cudaSetDevice(g->device));
    CRT_CUDA(cudaFree(g->nodes));
    CRT_CUDA(cudaFree(g->tris));
    if (g->node_box) CRT_CUDA(cudaFree(g->node_box));
    if (g->light_table) CRT_CUDA(cudaFree(g->light_table));
    if (g->light_scratch) CRT_CUDA(cudaFree(g->light_scratch));
    delete g;
    return CRT_OK;
}

extern "C" int crt_geometry_stats(crt_geometry g, double out[8])
{
    CRT_REQUIRE(g && out, "null argument");
    out[0] = (double)g->n_tris;
    out[1] = (double)g->n_nodes;
    out[2] = (double)g->max_depth;
    out[3] = (double)g->build_ms;
    out[4] = (double)(g->n_nodes * sizeof(WideNode));
    out[5] = (double)(g->n_tris * sizeof(WideTri));
    out[6] = (double)g->pad;
    out[7] = (double)g->refit_ms;
    return CRT_OK;
}

extern "C" int crt_trace_closest(crt_ctx* ctx, crt_geometry g, size_t n, const float* d_org, const float* d_dir,
                                 float tmin, float tmax, int32_t* d_out_prim, float* d_out_tuv)
{
    CRT_REQUIRE(ctx && g && d_org && d_dir && d_out_prim && d_out_tuv, "null argument");
    if (n == 0) return CRT_OK;
    k_trace<false><<<div_up(n, 256), 256, 0, ctx->stream>>>(g->view(), n, d_org, d_dir, tmin, tmax, d_out_prim,
                                                           d_out_tuv);
    return check_launch(ctx, "trace_closest");
}

extern "C" int crt_trace_any(crt_ctx* ctx, crt_geometry g, size_t n, const float* d_org, const float* d_dir,
                             float tmin, float tmax, int32_t* d_out_hit)
{
    CRT_REQUIRE(ctx && g && d_org && d_dir && d_out_hit, "null argument");
    if (n == 0) return CRT_OK;
    k_trace<true><<<div_up(n, 256), 256, 0, ctx->stream>>>(g->view(), n, d_org, d_dir, tmin, tmax, d_out_hit, nullptr);
    return check_launch(ctx, "trace_any");
}

extern "C" int crt_trace_closest_brute(crt_ctx* ctx, const crt_triangle* d_triangles, size_t n_tris, size_t n,
                                       const float* d_org, const float* d_dir, float tmin, float tmax,
                                       int32_t* d_out_prim, float* d_out_tuv)
{
    CRT_REQUIRE(ctx && d_org && d_dir && d_out_prim && d_out_tuv, "null argument");
    CRT_REQUIRE(n_tris == 0 || d_triangles, "null triangle array");
    if (n == 0) return CRT_OK;
    k_trace_brute<<<div_up(n * 32, 256), 256, 0, ctx->stream>>>((const float*)d_triangles, (uint32_t)n_tris, n, d_org,
                                                               d_dir, tmin, tmax, d_out_prim, d_out_tuv);
    return check_launch(ctx, "trace_closest_brute");
}
