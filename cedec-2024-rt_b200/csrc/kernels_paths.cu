// kernels_paths.cu — examples 07_pt / 08_nee / 09_ris (07_pt.cu:11-90, 08_nee.cu:11-129, 09_ris.cu:11-166) as a wavefront.
//
// The reference traces a whole path inside one kernel: closest hit, light sampling with its shadow rays, bounce, up to
// max_depth times.  As a single CUDA kernel with the per-thread walk that runs at 4-8 lanes per instruction
// (profiles/r2/ncu_r2_cfg_summary.csv): lanes wait for the longest walk of every ray, and 09_ris with the shadowed target
// function walks 33 shadow rays per path vertex one after the other.  Here a frame is, per path depth,
//
//   k_pt_emit_closest + k_trace_closest_queue   the closest hit of every live path's ray: ray records and the persistent
//                       pooled closest-hit kernel of shadow_queue.cuh (k_pt_closest, the per-thread walk, with CRT_POOLED_CLOSEST=0)
//   k_pt_vertex         miss / emitter / surface; light sampling; the shadow rays are only *emitted*: compact 32-byte
//                       records, one queue reservation per warp, ray c of the warp's paths next to each other
//   k_trace_shadow_queue<kEpiBitmask>   the persistent any-hit kernel of shadow_queue.cuh: bit c of the path's mask = ray c
//                       is unoccluded
//   k_pt_replay         09_ris with use_shadowed_target_function only: the 32 candidates again from the saved random
//                       state, now with their visibilities (Reservoir::update in the reference's order), then the ray
//                       towards the selected sample — traced by a second k_trace_shadow_queue launch
//   k_pt_shade_bounce   radiance of the vertex, next direction, throughput
//
// and k_pt_begin / k_pt_write around the loop.  Per path the random numbers, their order and every arithmetic
// operation are those of px_path_trace (restir_pixel.cuh), which stays as the single-kernel form (CRT_WAVEFRONT=0, and the
// host emulation of tests/emu); results are bit-identical (tests/test_gpu_parity.py, tests/test_gpu_configs.py).
// One shadow ray fewer than the reference per vertex of the shadowed 09_ris: its final target function repeats
// check_visibility with the arguments of the visibility ray just traced (09_ris.cu:112,116-119) — a pure function, traced once.
#include "launch_common.cuh"

namespace crt
{
// per-path state, one entry per pixel of the image (pixel_idx order); pointers into one allocation of the context
struct PathState
{
    unsigned long long* rng;       // Pcg::state (sequence 0: inc == 1)
    unsigned long long* rng_snap;  // the state before this vertex's light sampling (k_pt_replay / k_pt_shade_bounce redraw from it)
    float4* ro_t;                  // ray origin, hit distance
    float4* rd_prim;               // ray direction, hit primitive id (int bits): kPathDead / -1 (miss or not traced yet) / id
    float4* thr;                   // throughput
    float4* rad;                   // radiance
    float4* sel0;                  // 09_ris: selected sample — hit_position.xyz, w_sum
    float4* sel1;                  //         hit_normal.xyz, M (int bits)
    float4* sel2;                  //         radiance.xyz
    uint32_t* vmask;               // bit c: shadow ray c of this vertex is unoccluded
    uint32_t* vfinal;              // shadowed 09_ris: bit 0: the ray towards the selected sample is unoccluded
};
constexpr int kPathDead = -2;
constexpr size_t kPathStateBytes = 8 + 8 + 16 * 7 + 4 + 4;

__device__ __forceinline__ Pcg pcg_from_state(unsigned long long state)
{
    Pcg r(0, 0);
    r.state = state;
    r.inc = 1u;
    return r;
}
__device__ __forceinline__ f3 xyz(float4 v) { return f3{v.x, v.y, v.z}; }

__global__ void __launch_bounds__(256)
    k_pt_begin(int W, int H, Rows rows, int frame, crt_raygen raygen, PathState st)
{
    const TilePix t = this_pixel(W, H, rows);
    if (!t.in) return;
    const Pix px = t.px;
    Pcg rng(hash_pcg3(px.xi, px.yi, frame), 0);
    f3 ro, rd;
    primary_ray(raygen, px, W, H, ro, rd);
    st.rng[px.idx] = rng.state;
    st.ro_t[px.idx] = make_float4(ro.x, ro.y, ro.z, 0.0f);
    st.rd_prim[px.idx] = make_float4(rd.x, rd.y, rd.z, __int_as_float(-1));
    st.thr[px.idx] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
    st.rad[px.idx] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}

__global__ void __launch_bounds__(256)
    k_pt_closest(int W, int H, Rows rows, Bvh bvh, PathState st, unsigned long long* ray_counters)
{
    const TilePix t = this_pixel(W, H, rows);
    bool traced = false;
    if (t.in)
    {
        const int idx = t.px.idx;
        const float4 rdp = st.rd_prim[idx];
        if (__float_as_int(rdp.w) != kPathDead)
        {
            const float4 rot = st.ro_t[idx];
            Hit h;
            trace<false>(bvh, xyz(rot), xyz(rdp), 0.0f, kFltMax, h);
            st.ro_t[idx].w = h.t;
            st.rd_prim[idx].w = __int_as_float(h.prim);
            traced = true;
        }
    }
    const uint32_t c = __reduce_add_sync(0xffffffffu, traced ? 1u : 0u);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(ray_counters + 0, (unsigned long long)c);
}

// the live paths' rays as queue records for k_trace_closest_queue (shadow_queue.cuh)
__global__ void __launch_bounds__(256)
    k_pt_emit_closest(int W, int H, Rows rows, PathState st, ShadowQueue q, unsigned long long* ray_counters)
{
    const TilePix t = this_pixel(W, H, rows);
    const int idx = t.px.idx;
    float4 rdp = make_float4(0, 0, 0, 0);
    bool live = false;
    if (t.in)
    {
        rdp = st.rd_prim[idx];
        live = __float_as_int(rdp.w) != kPathDead;
    }
    // one reservation per block (two same-address atomics per warp made this kernel wait for the L2's atomic unit)
    __shared__ uint32_t s_cnt[8], s_base;
    const unsigned mask = __ballot_sync(0xffffffffu, live);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) s_cnt[warp] = (uint32_t)__popc(mask);
    __syncthreads();
    if (threadIdx.x == 0)
    {
        uint32_t total = 0;
#pragma unroll
        for (int w = 0; w < 8; w++)
        {
            const uint32_t c = s_cnt[w];
            s_cnt[w] = total;
            total += c;
        }
        s_base = total ? atomicAdd(q.count, total) : 0u;
        if (total) atomicAdd(ray_counters + 0, (unsigned long long)total);
    }
    __syncthreads();
    if (!live) return;
    const float4 rot = st.ro_t[idx];
    float4* dst = (float4*)q.rays + ((size_t)s_base + s_cnt[warp] + (size_t)__popc(mask & ((1u << lane) - 1u))) * 2;
    dst[0] = make_float4(rot.x, rot.y, rot.z, __uint_as_float((uint32_t)idx));
    dst[1] = make_float4(rdp.x, rdp.y, rdp.z, 0.0f);
}

// compact ray record of path `pix`, ray `c` of its vertex (the tracer's kEpiBitmask epilogue sets bit c)
__device__ __forceinline__ void put_ray(const ShadowQueue& q, uint32_t slot, f3 org, f3 dir, uint32_t pix, uint32_t c)
{
    float4* dst = (float4*)q.rays + (size_t)slot * 2;
    dst[0] = make_float4(org.x, org.y, org.z, __uint_as_float(pix | (c << 27)));
    dst[1] = make_float4(dir.x, dir.y, dir.z, 0.0f);
}
// a reserved record no ray was written to (kHoleRecord, shadow_queue.cuh): the tracer fetches and drops it
__device__ __forceinline__ void put_hole(const ShadowQueue& q, uint32_t slot)
{
    ((float4*)q.rays)[(size_t)slot * 2] = make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(kHoleRecord));
}
// check_visibility's segment against the triangle it starts on; -DCRT_NO_OWN_TRI: never (A/B)
__device__ __forceinline__ bool own_triangle_stops(f3 org, f3 dir, const TriRef& own)
{
#if defined(CRT_NO_OWN_TRI)
    return false;
#else
    return segment_hits_triangle(org, dir, 0.0f, 0.99f, own.v(0), own.v(1), own.v(2));
#endif
}
// every lane of the warp calls this: reserves rays_per_path slots for each lane that emits; returns the lane's first slot
// and the stride between its consecutive rays (ray c of the warp's emitting paths lie next to each other)
__device__ __forceinline__ uint32_t reserve_rays(const ShadowQueue& q, bool emits, uint32_t rays_per_path, uint32_t& stride)
{
    const unsigned mask = __ballot_sync(0xffffffffu, emits);
    stride = (uint32_t)__popc(mask);
    if (mask == 0) return 0;
    const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(q.count, stride * rays_per_path);
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + (uint32_t)__popc(mask & ((1u << lane) - 1u));
}

// EX 7 / 8 / 9: the vertex of every live path after its closest-hit walk (07_pt.cu:36-70, 08_nee.cu:40-80, 09_ris.cu:40-100)
// LS: the light source — LightsIndexed over the reference's light list (uniform selection) or LightsTable over the slot
// table of power-proportional selection (n_lights = K, restir_core.cuh)
template <int EX, int MODE, class LS>
__global__ void __launch_bounds__(256)
    k_pt_vertex(int W, int H, Rows rows, int depth, Bvh bvh, const float* tris60, const typename LS::Elem* lights, uint32_t n_lights,
                crt_options options, PathState st, ShadowQueue q, unsigned long long* ray_counters)
{
    const TilePix t = this_pixel(W, H, rows);
    const Opt opt = make_opt(options);
    const int idx = t.px.idx;
    bool lit = false;  // this path samples a light at this vertex
    float4 rot = make_float4(0, 0, 0, 0), rdp = rot;
    int prim = kPathDead;
    if (t.in)
    {
        rdp = st.rd_prim[idx];
        prim = __float_as_int(rdp.w);
    }
    f3 color{0, 0, 0};
    Surf surf{{0, 0, 0}, {0, 0, 0}};
    if (prim != kPathDead)
    {
        rot = st.ro_t[idx];
        const f3 thr = xyz(st.thr[idx]);
        if (prim < 0)
        {
            if (EX == 7)
            {
                const f3 r = xyz(st.rad[idx]) + thr * opt.sky;
                st.rad[idx] = make_float4(r.x, r.y, r.z, 0.0f);
            }
            st.rd_prim[idx].w = __int_as_float(kPathDead);
        }
        else
        {
            const TriRef tri = tri_at(tris60, prim);
            const f3 em = tri.emissive();
            if (has_emission(em))
            {
                if (EX == 7 || depth == 0)
                {
                    const f3 r = xyz(st.rad[idx]) + thr * em;
                    st.rad[idx] = make_float4(r.x, r.y, r.z, 0.0f);
                }
                st.rd_prim[idx].w = __int_as_float(kPathDead);
            }
            else
            {
                surf = surface_from_hit(tri, xyz(rot), xyz(rdp), rot.w);
                color = tri.color();
                lit = EX != 7;
                if (EX == 7)
                {
                    // naive path tracing: straight to the bounce (07_pt.cu:72-85)
                    Pcg rng = pcg_from_state(st.rng[idx]);
                    const f3 wo = bounce_direction<Math<MODE>>(surf, tri, rng);
                    const f3 nt = thr * color, no = surf.p + 0.001f * surf.n;
                    st.rng[idx] = rng.state;
                    st.thr[idx] = make_float4(nt.x, nt.y, nt.z, 0.0f);
                    st.ro_t[idx] = make_float4(no.x, no.y, no.z, 0.0f);
                    st.rd_prim[idx] = make_float4(wo.x, wo.y, wo.z, __int_as_float(-1));
                }
            }
        }
    }
    if (EX == 7) return;
    const bool shadowed = EX == 9 && opt.shadowed;
    const LS L = LS::at(tris60, lights, n_lights);
    const f3 org = surf.p + 0.001f * surf.n;  // check_visibility's segment (raytrace.hpp:45-52): direction p1 - p0, t in [0, 0.99]
    Pcg rng(0, 0);
    if (lit)
    {
        rng = pcg_from_state(st.rng[idx]);
        st.rng_snap[idx] = rng.state;
        st.vmask[idx] = 0u;
    }
    // Own-triangle pre-test (segment_hits_triangle, bvh.cuh): a light sample below the horizon of the triangle the vertex
    // lies on — about half of the uniformly drawn candidates — is stopped by that triangle; the ray is decided here
    // (its visibility bit stays 0) instead of being walked through the tree.
    uint32_t traced = 0;  // rays this lane hands to the tracer
    if (!shadowed)
    {
        f3 dir{0, 0, 0};
        bool emits = false;
        if (lit)
        {
            if (EX == 8)
            {
                const float r0 = rng.next_f();
                const float r1 = rng.next_f();
                const float r2 = rng.next_f();
                const LightSample ls = L.sample(r0, r1, r2);
                dir = ls.p - surf.p;
            }
            else
            {
                // 09_ris.cu:66-100 with the unshadowed target function: the reservoir is final here
                const Res r = ris_candidates(bvh, L, surf, opt.ris_count, false, rng);
                st.sel0[idx] = make_float4(r.s.hp.x, r.s.hp.y, r.s.hp.z, r.w_sum);
                st.sel1[idx] = make_float4(r.s.hn.x, r.s.hn.y, r.s.hn.z, __int_as_float(r.M));
                st.sel2[idx] = make_float4(r.s.rad.x, r.s.rad.y, r.s.rad.z, 0.0f);
                dir = r.s.hp - surf.p;
            }
            st.rng[idx] = rng.state;
            emits = !own_triangle_stops(org, dir, tri_at(tris60, prim));
        }
        // one reservation and one update of each ray counter per block (three same-address atomics per warp made this kernel
        // wait for the L2's atomic unit: a launch is ~0.1 ms long and has 65 k warps)
        __shared__ uint32_t s_cnt[8], s_dec[8], s_base;
        const unsigned mask = __ballot_sync(0xffffffffu, emits), dmask = __ballot_sync(0xffffffffu, lit && !emits);
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (lane == 0)
        {
            s_cnt[warp] = (uint32_t)__popc(mask);
            s_dec[warp] = (uint32_t)__popc(dmask);
        }
        __syncthreads();
        if (threadIdx.x == 0)
        {
            uint32_t total = 0, dec = 0;
#pragma unroll
            for (int w = 0; w < 8; w++)
            {
                const uint32_t c = s_cnt[w];
                s_cnt[w] = total;
                total += c;
                dec += s_dec[w];
            }
            s_base = total ? atomicAdd(q.count, total) : 0u;
            if (total) atomicAdd(ray_counters + 1, (unsigned long long)total);
            if (dec) atomicAdd(ray_counters + 2, (unsigned long long)dec);  // crt_rays_decided_at_emission
        }
        __syncthreads();
        if (emits) put_ray(q, s_base + s_cnt[warp] + (uint32_t)__popc(mask & ((1u << lane) - 1u)), org, dir, (uint32_t)idx, 0u);
        return;  // counted above
    }
    else
    {
        // one shadow ray per candidate; k_pt_replay draws the same candidates again once their visibilities are known.
        // The warp reserves ris_count rows of `stride` records; a lane fills its column from the top with the rays that
        // need a walk and marks the rest of the column as holes, which the tracer skips when it fetches them.
        const uint32_t per_path = (uint32_t)(opt.ris_count > 0 ? opt.ris_count : 0);
        uint32_t stride = 0;
        const uint32_t slot = reserve_rays(q, lit && per_path > 0, per_path, stride);
        if (lit)
        {
            const TriRef own = tri_at(tris60, prim);
            for (int c = 0; c < opt.ris_count; ++c)
            {
                const float r0 = rng.next_f();
                const float r1 = rng.next_f();
                const float r2 = rng.next_f();
                (void)rng.next_f();  // the reservoir's u of this candidate
                const LightSample ls = L.sample(r0, r1, r2);
                const f3 dir = ls.p - surf.p;
                if (own_triangle_stops(org, dir, own)) continue;
                put_ray(q, slot + traced * stride, org, dir, (uint32_t)idx, (uint32_t)c);
                ++traced;
            }
            for (uint32_t j = traced; j < per_path; ++j) put_hole(q, slot + j * stride);
            st.rng[idx] = rng.state;
        }
    }
    const uint32_t wanted = lit ? (shadowed ? (uint32_t)(opt.ris_count > 0 ? opt.ris_count : 0) : 1u) : 0u;
    const uint32_t n_traced = __reduce_add_sync(0xffffffffu, traced), n_decided = __reduce_add_sync(0xffffffffu, wanted - traced);
    if ((threadIdx.x & 31) == 0)
    {
        if (n_traced) atomicAdd(ray_counters + 1, (unsigned long long)n_traced);
        if (n_decided) atomicAdd(ray_counters + 2, (unsigned long long)n_decided);  // crt_rays_decided_at_emission
    }
}

// shadowed 09_ris: Reservoir::update over the candidates with their visibilities, then the ray towards the selected sample
template <int MODE, class LS>
__global__ void __launch_bounds__(256)
    k_pt_replay(int W, int H, Rows rows, Bvh bvh, const float* tris60, const typename LS::Elem* lights, uint32_t n_lights, crt_options options,
                PathState st, ShadowQueue q, unsigned long long* ray_counters)
{
    const TilePix t = this_pixel(W, H, rows);
    const Opt opt = make_opt(options);
    const int idx = t.px.idx;
    int prim = kPathDead;
    if (t.in) prim = __float_as_int(st.rd_prim[idx].w);
    const bool lit = prim >= 0;  // k_pt_vertex killed the paths that missed or hit an emitter
    uint32_t stride = 0;
    const uint32_t slot = reserve_rays(q, lit, 1u, stride);
    const uint32_t n_emit = __reduce_add_sync(0xffffffffu, lit ? 1u : 0u);
    if ((threadIdx.x & 31) == 0 && n_emit) atomicAdd(ray_counters + 1, (unsigned long long)n_emit);
    if (!lit) return;
    const float4 rot = st.ro_t[idx], rdp = st.rd_prim[idx];
    const TriRef tri = tri_at(tris60, prim);
    const Surf surf = surface_from_hit(tri, xyz(rot), xyz(rdp), rot.w);
    const LS L = LS::at(tris60, lights, n_lights);
    Pcg rng = pcg_from_state(st.rng_snap[idx]);
    const uint32_t vmask = st.vmask[idx];
    Res r = empty_res();
    const float inv_n = 1.0f / (float)n_lights;
    for (int c = 0; c < opt.ris_count; ++c)
    {
        const float r0 = rng.next_f();
        const float r1 = rng.next_f();
        const float r2 = rng.next_f();
        const float u = rng.next_f();
        const LightSample ls = L.sample(r0, r1, r2);
        // target function with visibility, in the reference's order: ((1/pi * G) * V) * luminance (reservoir.hpp:42-59)
        const float V = ((vmask >> c) & 1u) ? 1.0f : 0.0f;
        const float p_hat = kInvPi * geometry_term(surf.p, surf.n, ls.p, ls.n) * V * luminance(ls.emissive);
        if (LS::kHasPdf) ris_apply_pdf(surf, ls, ls.pdf, u, p_hat, r);
        else ris_apply(surf, ls, inv_n, u, p_hat, r);
    }
    st.sel0[idx] = make_float4(r.s.hp.x, r.s.hp.y, r.s.hp.z, r.w_sum);
    st.sel1[idx] = make_float4(r.s.hn.x, r.s.hn.y, r.s.hn.z, __int_as_float(r.M));
    st.sel2[idx] = make_float4(r.s.rad.x, r.s.rad.y, r.s.rad.z, 0.0f);
    st.vfinal[idx] = 0u;
    put_ray(q, slot, surf.p + 0.001f * surf.n, r.s.hp - surf.p, (uint32_t)idx, 0u);
}

// 08_nee.cu:66-106 / 09_ris.cu:102-150: the vertex's radiance with the traced visibility, then the bounce
template <int EX, int MODE, class LS>
__global__ void __launch_bounds__(256)
    k_pt_shade_bounce(int W, int H, Rows rows, Bvh bvh, const float* tris60, const typename LS::Elem* lights, uint32_t n_lights,
                      crt_options options, PathState st)
{
    const TilePix t = this_pixel(W, H, rows);
    if (!t.in) return;
    const Opt opt = make_opt(options);
    const int idx = t.px.idx;
    const float4 rdp = st.rd_prim[idx];
    const int prim = __float_as_int(rdp.w);
    if (prim < 0) return;
    const float4 rot = st.ro_t[idx];
    const TriRef tri = tri_at(tris60, prim);
    const Surf surf = surface_from_hit(tri, xyz(rot), xyz(rdp), rot.w);
    const f3 color = tri.color();
    const f3 thr = xyz(st.thr[idx]);
    f3 radiance = xyz(st.rad[idx]);
    const bool shadowed = EX == 9 && opt.shadowed;
    if (EX == 8)
    {
        Pcg rs = pcg_from_state(st.rng_snap[idx]);
        const float r0 = rs.next_f();
        const float r1 = rs.next_f();
        const float r2 = rs.next_f();
        const LightSample ls = LS::at(tris60, lights, n_lights).sample(r0, r1, r2);
        const float V = (st.vmask[idx] & 1u) ? 1.0f : 0.0f;
        const f3 brdf = kInvPi * color;
        const float G = geometry_term(surf.p, surf.n, ls.p, ls.n);
        const float light_pdf = light_pdf_of<LS>(ls, n_lights);
        radiance = radiance + thr * brdf * G * V * ls.emissive / light_pdf;
    }
    else
    {
        const float4 s0 = st.sel0[idx], s1 = st.sel1[idx], s2 = st.sel2[idx];
        Res r = empty_res();
        r.s.hp = xyz(s0);
        r.s.hn = xyz(s1);
        r.s.rad = xyz(s2);
        r.w_sum = s0.w;
        r.M = __float_as_int(s1.w);
        const float V = ((shadowed ? st.vfinal[idx] : st.vmask[idx]) & 1u) ? 1.0f : 0.0f;
        const f3 brdf = kInvPi * color;
        const float G = geometry_term(surf.p, surf.n, r.s.hp, r.s.hn);
        // target_function(..., use_shadowed_target_function): ((1/pi * G) * V) * luminance with the very V above
        const float p_hat = shadowed ? kInvPi * geometry_term(surf.p, surf.n, r.s.hp, r.s.hn) * V * luminance(r.s.rad)
                                     : kInvPi * geometry_term(surf.p, surf.n, r.s.hp, r.s.hn) * luminance(r.s.rad);
        radiance = radiance + thr * brdf * G * V * r.s.rad * ucw_of(r, p_hat);
    }
    Pcg rng = pcg_from_state(st.rng[idx]);
    const f3 wo = bounce_direction<Math<MODE>>(surf, tri, rng);
    const f3 nt = thr * color, no = surf.p + 0.001f * surf.n;  // offset_ray_position, core.hpp:32-36
    st.rng[idx] = rng.state;
    st.rad[idx] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
    st.thr[idx] = make_float4(nt.x, nt.y, nt.z, 0.0f);
    st.ro_t[idx] = make_float4(no.x, no.y, no.z, 0.0f);
    st.rd_prim[idx] = make_float4(wo.x, wo.y, wo.z, __int_as_float(-1));
}

__global__ void __launch_bounds__(256) k_pt_write(int W, int H, Rows rows, PathState st, crt_float4* accum, int accumulate)
{
    const TilePix t = this_pixel(W, H, rows);
    if (t.in) write_accum(accum, t.px.idx, xyz(st.rad[t.px.idx]), accumulate != 0);
}

static int path_state(crt_ctx* ctx, size_t n, PathState* st)
{
    if (ctx->path_state_pixels < n)
    {
        if (ctx->path_state) CRT_CUDA(cudaFree(ctx->path_state));
        ctx->path_state = nullptr;
        ctx->path_state_pixels = 0;
        CRT_CUDA(cudaMalloc(&ctx->path_state, n * kPathStateBytes + 256));
        ctx->path_state_pixels = n;
    }
    const size_t cap = ctx->path_state_pixels;
    char* p = (char*)ctx->path_state;
    st->ro_t = (float4*)p; p += cap * 16;
    st->rd_prim = (float4*)p; p += cap * 16;
    st->thr = (float4*)p; p += cap * 16;
    st->rad = (float4*)p; p += cap * 16;
    st->sel0 = (float4*)p; p += cap * 16;
    st->sel1 = (float4*)p; p += cap * 16;
    st->sel2 = (float4*)p; p += cap * 16;
    st->rng = (unsigned long long*)p; p += cap * 8;
    st->rng_snap = (unsigned long long*)p; p += cap * 8;
    st->vmask = (uint32_t*)p; p += cap * 4;
    st->vfinal = (uint32_t*)p;
    return CRT_OK;
}

template <int EX, int MODE, class LS>
static int path_trace_wavefront_impl(crt_ctx* ctx, int W, int H, int frame, crt_geometry geom, const float* tris60,
                                     const typename LS::Elem* lights, uint32_t n_lights, crt_raygen raygen, crt_options options,
                                     crt_float4* accum, unsigned long long* counters)
{
    const Rows all = rows_of(ctx, H);
    const bool shadowed = EX == 9 && options.use_shadowed_target_function != 0;
    const size_t rays_per_px = shadowed ? (size_t)(options.ris_sample_count > 0 ? options.ris_sample_count : 0) : 1;
    // bands of rows, so that a band's ray queue (pixels x rays x 32 B) stays below 4 GiB
    const size_t per_row = (size_t)W * (rays_per_px ? rays_per_px : 1) * 32u;
    int band = (int)(((size_t)4 << 30) / per_row);
    band = band < kTileH ? kTileH : band / kTileH * kTileH;
    PathState st;
    int rc = path_state(ctx, (size_t)W * H, &st);
    if (rc != CRT_OK) return rc;
    const Bvh bvh = geom->view();
    for (int y0 = all.y0; y0 < all.y1; y0 += band)
    {
        const Rows rows{y0, y0 + band < all.y1 ? y0 + band : all.y1};
        const dim3 grid = tile_grid(W, rows);
        const size_t n_px = (size_t)(rows.y1 - rows.y0) * W;
        CRT_REQUIRE(n_px * (rays_per_px ? rays_per_px : 1) < 0x07ffffffull * 32ull, "too many shadow rays in one band");
        CRT_REQUIRE((size_t)W * H < 0x07ffffffull, "image too large for the packed path | ray word");
        k_pt_begin<<<grid, 256, 0, ctx->stream>>>(W, H, rows, frame, raygen, st);
        rc = check_launch(ctx, "pt_begin");
        for (int depth = 0; rc == CRT_OK && depth < options.max_depth; ++depth)
        {
            ShadowQueue q{nullptr, nullptr, nullptr, 0};
            // closest hits: the persistent pooled kernel for the incoherent bounce rays, the per-thread walk for the coherent
            // camera rays (08_nee at 1080p: 2.74 ms per frame; pooled for every depth 2.88; per-thread for every depth 3.61 —
            // profiles/r2/tuning.txt).  CRT_POOLED_CLOSEST = 0 never / 1 bounce rays (default) / 2 always
            if (ctx->pooled_closest >= (depth == 0 ? 2 : 1))
            {
                rc = queue_prepare(ctx, (n_px + 1) / 2, &q);
                if (rc != CRT_OK) break;
                q.stride4 = 2;
                k_pt_emit_closest<<<grid, 256, 0, ctx->stream>>>(W, H, rows, st, q, counters);
                rc = check_launch(ctx, "pt_emit_closest");
                if (rc != CRT_OK) break;
                static int closest_blocks = 0;
                if (!closest_blocks)
                {
                    CRT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&closest_blocks, k_trace_closest_queue, kShadowWarps * 32, 0));
                    if (closest_blocks < 1) closest_blocks = 1;
                }
                k_trace_closest_queue<<<closest_blocks * ctx->sm_count, kShadowWarps * 32, 0, ctx->stream>>>(bvh, q, ClosestSink{st.ro_t, st.rd_prim});
                rc = check_launch(ctx, "trace_closest");
            }
            else
            {
                k_pt_closest<<<grid, 256, 0, ctx->stream>>>(W, H, rows, bvh, st, counters);
                rc = check_launch(ctx, "pt_closest");
            }
            if (rc != CRT_OK) break;
            if (EX != 7)
            {
                rc = queue_prepare(ctx, (n_px * (rays_per_px ? rays_per_px : 1) + 1) / 2, &q);  // capacity in 64-byte records
                if (rc != CRT_OK) break;
                q.stride4 = 2;
            }
            k_pt_vertex<EX, MODE, LS><<<grid, 256, 0, ctx->stream>>>(W, H, rows, depth, bvh, tris60, lights, n_lights, options, st, q, counters);
            rc = check_launch(ctx, "pt_vertex");
            if (rc != CRT_OK || EX == 7) continue;
            ShadowSink sink{nullptr, nullptr, 0, nullptr};
            sink.visible_count = st.vmask;
            rc = queue_trace<kEpiBitmask>(ctx, geom, q, sink);
            if (rc != CRT_OK) break;
            if (shadowed)
            {
                rc = queue_prepare(ctx, (n_px + 1) / 2, &q);
                if (rc != CRT_OK) break;
                q.stride4 = 2;
                k_pt_replay<MODE, LS><<<grid, 256, 0, ctx->stream>>>(W, H, rows, bvh, tris60, lights, n_lights, options, st, q, counters);
                rc = check_launch(ctx, "pt_replay");
                if (rc != CRT_OK) break;
                sink.visible_count = st.vfinal;
                rc = queue_trace<kEpiBitmask>(ctx, geom, q, sink);
                if (rc != CRT_OK) break;
            }
            k_pt_shade_bounce<EX, MODE, LS><<<grid, 256, 0, ctx->stream>>>(W, H, rows, bvh, tris60, lights, n_lights, options, st);
            rc = check_launch(ctx, "pt_shade_bounce");
        }
        if (rc != CRT_OK) return rc;
        k_pt_write<<<grid, 256, 0, ctx->stream>>>(W, H, rows, st, accum, options.accumulate);
        rc = check_launch(ctx, "pt_write");
        if (rc != CRT_OK) return rc;
    }
    return CRT_OK;
}

int path_trace_wavefront(crt_ctx* ctx, int example, int W, int H, int frame, crt_geometry geom, const float* tris60,
                         const uint32_t* lights, uint32_t n_lights, const LightRec* slots, uint32_t n_slots, crt_raygen raygen,
                         crt_options options, crt_float4* accum, unsigned long long* counters)
{
    const bool ex = ctx->math_mode == CRT_MATH_EXACT;
#define CRT_PT_LS(EX, LS, P, N) (ex ? path_trace_wavefront_impl<EX, 1, LS>(ctx, W, H, frame, geom, tris60, P, N, raygen, options, accum, counters) \
                                    : path_trace_wavefront_impl<EX, 0, LS>(ctx, W, H, frame, geom, tris60, P, N, raygen, options, accum, counters))
#define CRT_PT(EX) (slots ? CRT_PT_LS(EX, LightsTable, slots, n_slots) : CRT_PT_LS(EX, LightsIndexed, lights, n_lights))
    if (example == 7) return CRT_PT_LS(7, LightsIndexed, lights, n_lights);
    if (example == 8) return CRT_PT(8);
    return CRT_PT(9);
#undef CRT_PT
#undef CRT_PT_LS
}
}  // namespace crt
