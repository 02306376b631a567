// restir_pixel.cuh — the per-pixel bodies of the reference's kernels, independent of thread mapping and of
// how reservoirs are stored.  `RS` is a reservoir store with load(idx) / store(idx, Res): AosStore is the
// reference's 76-byte AoS layout (drop-in mode), SoaStore (kernels_fast.cu) the planar fast path.
// Host-callable so that tests/emu can run the very same bodies on the CPU against the oracle.
#pragma once
#include "../../include/cedecrt.h"
#include "restir_core.cuh"

namespace crt
{
struct Pix
{
    int xi, yi, idx;  // buffers are stored bottom-up: idx = xi + (H - yi - 1) * W (10_restir_di.cu:18-20)
};
CRT_HD Pix make_pix(int xi, int yi, int W, int H) { return Pix{xi, yi, xi + (H - yi - 1) * W}; }

struct Vis
{
    float u, v;
    int index;
};
CRT_HD Vis load_vis(const crt_visibility* buf, int idx)
{
    const u4 q = load_u4(buf + idx);
    return {u2f(q.x), u2f(q.y), (int)q.z};
}
CRT_HD void store_vis(crt_visibility* buf, int idx, const Hit& h)
{
    // Visibility{isect.uv, isect.index}: a miss leaves uv = (0,0), index = -1; _pad = 0
    crt_visibility v;
    v.uv[0] = h.prim < 0 ? 0.0f : h.u;
    v.uv[1] = h.prim < 0 ? 0.0f : h.v;
    v.index = h.prim;
    v._pad = 0;
#if defined(__CUDA_ARCH__)
    *((float4*)(buf + idx)) = make_float4(v.uv[0], v.uv[1], __int_as_float(v.index), 0.0f);
#else
    buf[idx] = v;
#endif
}

// Reservoir, 76 bytes = 19 words (common/reservoir.hpp:5-38); word 15 holds `bool visibility` in its low byte
struct AosStore
{
    crt_reservoir* buf;
    CRT_HD Res load(int idx) const
    {
        const float* p = (const float*)(buf + idx);
        Res r;
        r.s.op = {p[0], p[1], p[2]};
        r.s.on = {p[3], p[4], p[5]};
        r.s.hp = {p[6], p[7], p[8]};
        r.s.hn = {p[9], p[10], p[11]};
        r.s.rad = {p[12], p[13], p[14]};
        r.s.vis = (f2u(p[15]) & 0xffu) ? 1u : 0u;
        r.w_sum = p[16];
        r.ucw = p[17];
        r.M = (int)f2u(p[18]);
        return r;
    }
    CRT_HD void store(int idx, const Res& r) const
    {
        float* p = (float*)(buf + idx);
        p[0] = r.s.op.x; p[1] = r.s.op.y; p[2] = r.s.op.z;
        p[3] = r.s.on.x; p[4] = r.s.on.y; p[5] = r.s.on.z;
        p[6] = r.s.hp.x; p[7] = r.s.hp.y; p[8] = r.s.hp.z;
        p[9] = r.s.hn.x; p[10] = r.s.hn.y; p[11] = r.s.hn.z;
        p[12] = r.s.rad.x; p[13] = r.s.rad.y; p[14] = r.s.rad.z;
        p[15] = u2f(r.s.vis & 1u);
        p[16] = r.w_sum;
        p[17] = r.ucw;
        p[18] = u2f((uint32_t)r.M);
    }
};

CRT_HD RayGen to_raygen(const crt_raygen& g)
{
    return RayGen{{g.m_origin.x, g.m_origin.y, g.m_origin.z},
                  {g.m_right.x, g.m_right.y, g.m_right.z},
                  {g.m_up.x, g.m_up.y, g.m_up.z}};
}
CRT_HD void primary_ray(const crt_raygen& raygen, const Pix& px, int W, int H, f3& ro, f3& rd)
{
    shoot(to_raygen(raygen), (float)px.xi / (float)W, (float)px.yi / (float)H, ro, rd);
}
// Moving geometry (crt_temporal_resampling_reprojected_motion, crt_restir_set_previous_triangles; DESIGN.md section 17):
// whether triangle `index` has other vertex bits (its 36 vertex bytes) in the previous frame's array than in this one's
CRT_HD bool tri_moved(const float* tris60, const float* prev_tris60, int index)
{
    const float* a = tris60 + (size_t)index * 15;
    const float* b = prev_tris60 + (size_t)index * 15;
    bool moved = false;
    for (int k = 0; k < 9; ++k) moved |= f2u(CRT_LDG(a + k)) != f2u(CRT_LDG(b + k));
    return moved;
}
// The point this surface point was at in the previous frame: the same barycentrics on the triangle's previous vertices,
// or `surf.p` itself when the triangle did not move (not a recomputation, which a contracted build may round otherwise)
CRT_HD f3 previous_point(const float* tris60, const float* prev_tris60, const Vis& v, const Surf& surf)
{
    if (!tri_moved(tris60, prev_tris60, v.index)) return surf.p;
    const TriRef pt = tri_at(prev_tris60, v.index);
    return bary_point(pt.v(0), pt.v(1), pt.v(2), v.u, v.v);
}
// The previous frame's primary-hit surface at pixel `idx`: its Visibility record and the eye that frame flipped the
// normal towards (its RayGenerator's origin: crt_raygen_lookat stores the eye).  False on a sky pixel.  Primary rays are
// deterministic, so this is the surface that frame's kernels used there when the geometry is static.  MOTION: the triangle
// is read from `prev_tris60`, the previous frame's array, when it moved (tri_moved) — only the pointer is chosen, so an
// unmoved triangle gives the static surface bit for bit.
template <bool MOTION = false>
CRT_HD bool previous_surface(const crt_visibility* prev_vis, const float* tris60, int idx, f3 prev_eye, Surf& s,
                             const float* prev_tris60 = nullptr)
{
    const Vis hv = load_vis(prev_vis, idx);
    if (hv.index == -1) return false;
    const float* t = MOTION && tri_moved(tris60, prev_tris60, hv.index) ? prev_tris60 : tris60;
    s = surface_from_visibility(tri_at(t, hv.index), hv.u, hv.v, prev_eye);
    return true;
}

// ---- 10_restir_di.cu:9-34
CRT_HD void px_raycast(const Pix& px, int W, int H, const Bvh& bvh, const crt_raygen& raygen, crt_visibility* vis)
{
    f3 ro, rd;
    primary_ray(raygen, px, W, H, ro, rd);
    Hit h;
    trace<false>(bvh, ro, rd, 0.0f, kFltMax, h);
    store_vis(vis, px.idx, h);
}
// The same with a HINT: the primitive id the Visibility record of this pixel holds before the call — last frame's answer
// when the host traces into the same buffer every frame, anything at all otherwise — names a triangle that is tested
// first, with the reference's own test on the tree's own vertex bits (`tris60` is the array the tree was built over), and
// a hit seeds the walk (bvh.cuh: trace_seeded).  The closest hit is decided by (t, primitive id) alone, so the stored
// record is the unhinted walk's bit for bit whatever the hint was; a good hint lets the walk cull with the final distance
// from its first node on (lab, config 5: 13.8 -> 12.0 node steps per primary ray with an unmoved camera).
CRT_HD void px_raycast_hinted(const Pix& px, int W, int H, const Bvh& bvh, const crt_raygen& raygen, crt_visibility* vis,
                              const float* tris60, uint32_t n_tris)
{
    f3 ro, rd;
    primary_ray(raygen, px, W, H, ro, rd);
    Hit h;
    h.prim = -1;
    h.t = kFltMax;
    h.u = h.v = 0.0f;
    const uint32_t old = (uint32_t)vis[px.idx].index;
    if (old < n_tris)
    {
        const TriRef tri = tri_at(tris60, (int)old);
        float t, u, v;
        if (ray_triangle(ro, rd, 0.0f, kFltMax, tri.v(0), tri.v(1), tri.v(2), t, u, v))
        {
            h.t = t;
            h.u = u;
            h.v = v;
            h.prim = (int)old;
        }
    }
    trace_seeded<false>(bvh, ro, rd, 0.0f, h);
    store_vis(vis, px.idx, h);
}

// A shadow ray the caller traces later (wavefront mode, shadow_queue.cuh): check_visibility's segment
// (raytrace.hpp:45-52) — origin p0 + 1e-3 n0, direction p1 - p0, t in [0, 0.99].
struct DeferredRay
{
    bool want;
    f3 org, dir;
    bool decided = false;  // the ray exists but needs no walk: the triangle it starts on stops it (visibility_ray_past_own)
};
CRT_HD DeferredRay visibility_ray(f3 p0, f3 n0, f3 p1) { return DeferredRay{true, p0 + 0.001f * n0, p1 - p0}; }
// The same ray, not wanted when the triangle it starts on stops it (segment_hits_triangle, bvh.cuh): the walk would
// report "occluded", which is what the caller has stored already.  -DCRT_NO_OWN_TRI traces every ray (A/B).
CRT_HD DeferredRay visibility_ray_past_own(f3 p0, f3 n0, f3 p1, const TriRef& own)
{
    DeferredRay r = visibility_ray(p0, n0, p1);
#if !defined(CRT_NO_OWN_TRI)
    if (segment_hits_triangle(r.org, r.dir, 0.0f, 0.99f, own.v(0), own.v(1), own.v(2)))
    {
        r.want = false;
        r.decided = true;
    }
#endif
    return r;
}

// ---- 10_restir_di.cu:36-135.  With `defer` the visibility-reuse ray is returned instead of traced and the
// reservoir is stored with visibility = false for the trace kernel to fill in.
template <class L, class RS>
CRT_HD DeferredRay px_generate_candidate(const Pix& px, int frame, const Bvh& bvh, const float* tris60,
                                         const crt_visibility* vis, f3 eye, const L& lights, const Opt& opt,
                                         const RS& out, bool defer = false)
{
    DeferredRay ray{false, {0, 0, 0}, {0, 0, 0}};
    const Vis v = load_vis(vis, px.idx);
    if (v.index == -1)
    {
        out.store(px.idx, empty_res());
        return ray;
    }
    const TriRef tri = tri_at(tris60, v.index);
    if (has_emission(tri.emissive()))
    {
        out.store(px.idx, empty_res());
        return ray;
    }
    Pcg rng(hash_pcg4(px.xi, px.yi, frame, 0), 0);
    const Surf surf = surface_from_visibility(tri, v.u, v.v, eye);
    Res r = ris_candidates(bvh, pixel_lights(lights, px.xi, px.yi, frame), surf, opt.ris_count, false, rng);
    r.ucw = ucw_of(r, target_function(bvh, surf.p, surf.n, r.s.hp, r.s.hn, r.s.rad, opt.shadowed));
    if (opt.reuse)
    {
        if (defer) ray = visibility_ray_past_own(surf.p, surf.n, r.s.hp, tri);  // r.s.vis is 0 = occluded here
        else r.s.vis = check_visibility(bvh, surf.p, surf.n, r.s.hp) != 0.0f ? 1u : 0u;
    }
    out.store(px.idx, r);
    return ray;
}

// ---- 10_restir_di.cu:137-237
// prev_cam != nullptr (extension: crt_temporal_resampling_reprojected): the previous reservoir is read at the pixel this
// surface point had in the previous frame's camera; no history there = Reservoir{} (restir_core.cuh: reproject_pixel)
// RW: CRT_REUSE_REFERENCE (the reference's merge) or CRT_REUSE_UNBIASED: temporal_merge_unbiased without a previous
// camera, temporal_merge_unbiased_reprojected with one — the history's surface is then the previous frame's at the
// history pixel, from `prev_vis` (the previous frame's Visibility buffer, read there only; unused by the reference's merge)
// MOTION (with a previous camera; crt_temporal_resampling_reprojected_motion): the look-up projects the point's previous
// position (previous_point on `prev_tris60`, the previous frame's triangle array) and the history's surface is built on
// the triangle the previous frame saw (previous_surface<true>)
template <class M, int RW = CRT_REUSE_REFERENCE, bool MOTION = false, class RSP, class RS>
CRT_HD void px_temporal(const Pix& px, int frame, const Bvh& bvh, const float* tris60, const crt_visibility* vis,
                        f3 eye, const Opt& opt, const RSP& prev, const RS& cur, const crt_raygen* prev_cam = nullptr,
                        int W = 0, int H = 0, const crt_visibility* prev_vis = nullptr, const float* prev_tris60 = nullptr)
{
    const Vis v = load_vis(vis, px.idx);
    if (v.index == -1) return;
    const TriRef tri = tri_at(tris60, v.index);
    if (has_emission(tri.emissive())) return;
    if (!opt.temporal) return;
    Pcg rng(hash_pcg4(px.xi, px.yi, frame, 1), 0);
    const Surf surf = surface_from_visibility(tri, v.u, v.v, eye);
    Res r = cur.load(px.idx);
    Res history;
    bool has_h = false;
    Surf hsurf{};
    if (prev_cam)
    {
        int xp, yp;
        const f3 p_prev = MOTION ? previous_point(tris60, prev_tris60, v, surf) : surf.p;
        const bool found = reproject_pixel(to_raygen(*prev_cam), W, H, p_prev, xp, yp);
        history = found ? prev.load(xp + (H - yp - 1) * W) : empty_res();
        if (RW == CRT_REUSE_UNBIASED && found && history.M > 0)
            has_h = previous_surface<MOTION>(prev_vis, tris60, xp + (H - yp - 1) * W, to_raygen(*prev_cam).origin, hsurf,
                                             prev_tris60);
    }
    else history = prev.load(px.idx);
    if (RW == CRT_REUSE_UNBIASED && prev_cam)
        temporal_merge_unbiased_reprojected<M>(bvh, surf, has_h, hsurf, eye, opt, history, r, rng);
    else if (RW == CRT_REUSE_UNBIASED) temporal_merge_unbiased<M>(bvh, surf, eye, opt, history, r, rng);
    else temporal_merge<M>(bvh, surf, eye, opt, history, r, rng);
    cur.store(px.idx, r);
}

// ---- 10_restir_di.cu:256-388
// RW = CRT_REUSE_UNBIASED: spatial_merge_unbiased with each accepted neighbour's surface (from its Visibility record),
// then a second pass over the same neighbours — the pixel's random stream replayed from before the loop: the same
// offsets, skips and one random number per visited neighbour — sums Z for the selected sample
template <class M, int RW = CRT_REUSE_REFERENCE, class RSI, class RSO>
CRT_HD void px_spatial(const Pix& px, int W, int H, int frame, int pass, const Bvh& bvh, const float* tris60,
                       const crt_visibility* vis, f3 eye, const Opt& opt, const RSI& in, const RSO& out)
{
    const Vis v = load_vis(vis, px.idx);
    if (v.index == -1) return;  // output left untouched, as in the reference
    const TriRef tri = tri_at(tris60, v.index);
    if (has_emission(tri.emissive())) return;
    Pcg rng(hash_pcg4(px.xi, px.yi, frame, 2 + pass), 0);
    const Surf surf = surface_from_visibility(tri, v.u, v.v, eye);
    Res r = in.load(px.idx);
    if (!opt.spatial)
    {
        out.store(px.idx, r);
        return;
    }
    const Pcg rng_z = rng;
    const int c_own = r.M;
    for (int k = 0; k < opt.spatial_count; ++k)
    {
        int x, y;
        spatial_neighbour<M>(px.xi, px.yi, opt.radius, rng, x, y);
        if (x < 0 || x >= W || y < 0 || y >= H) continue;
        if (x == px.xi && y == px.yi) continue;
        const int pid = x + (H - y - 1) * W;
        const Vis nv = load_vis(vis, pid);
        if (nv.index == -1) continue;
        const TriRef ntri = tri_at(tris60, nv.index);
        if (has_emission(ntri.emissive())) continue;
        if (RW == CRT_REUSE_UNBIASED)
            spatial_merge_unbiased<M>(bvh, surf, surface_from_visibility(ntri, nv.u, nv.v, eye), eye, opt, in.load(pid), r, rng);
        else spatial_merge<M>(bvh, surf, eye, opt, in.load(pid), r, rng);
    }
    const float p_hat = target_function(bvh, surf.p, surf.n, r.s.hp, r.s.hn, r.s.rad, opt.shadowed);
    if (RW != CRT_REUSE_UNBIASED) r.ucw = ucw_of(r, p_hat);
    else
    {
        int z = c_own;  // the pixel's own domain: ucw_unbiased reads p_hat_q(y) > 0 itself
        if (p_hat > 0.0f)
        {
            Pcg rz = rng_z;
            for (int k = 0; k < opt.spatial_count; ++k)
            {
                int x, y;
                spatial_neighbour<M>(px.xi, px.yi, opt.radius, rz, x, y);
                if (x < 0 || x >= W || y < 0 || y >= H) continue;
                if (x == px.xi && y == px.yi) continue;
                const int pid = x + (H - y - 1) * W;
                const Vis nv = load_vis(vis, pid);
                if (nv.index == -1) continue;
                const TriRef ntri = tri_at(tris60, nv.index);
                if (has_emission(ntri.emissive())) continue;
                const Surf ns = surface_from_visibility(ntri, nv.u, nv.v, eye);
                (void)rz.next_f();  // the merge's random number
                z = z_of(z, confidence<M>(in.load(pid).M, surf, ns, eye), bvh, ns, r.s, opt.shadowed);
            }
        }
        r.ucw = ucw_unbiased(r.w_sum, z, p_hat);
    }
    out.store(px.idx, r);
}

// ---- 10_restir_di.cu:390-459
CRT_HD void write_accum(crt_float4* accum, int idx, f3 c, bool add)
{
    crt_float4 a = {c.x, c.y, c.z, 1.0f};
    if (add)
    {
        const crt_float4 o = accum[idx];
        a = {o.x + c.x, o.y + c.y, o.z + c.z, o.w + 1.0f};
    }
    accum[idx] = a;
}
// With `shade` non-null the shadow ray is returned instead of traced, together with the factors of
// radiance = brdf * G * V * sample.radiance * ucw that the trace kernel multiplies out (shade->bg = brdf * G).
struct DeferredShade
{
    f3 bg, rad;
    float ucw;
};
template <class RS>
CRT_HD DeferredRay px_resolve(const Pix& px, crt_float4* accum, const Bvh& bvh, const float* tris60,
                              const crt_visibility* vis, f3 eye, const Opt& opt, const RS& res,
                              DeferredShade* shade = nullptr)
{
    DeferredRay ray{false, {0, 0, 0}, {0, 0, 0}};
    const Vis v = load_vis(vis, px.idx);
    if (v.index == -1)
    {
        accum[px.idx] = {0.0f, 0.0f, 0.0f, 1.0f};  // assigned even when accumulating
        return ray;
    }
    const TriRef tri = tri_at(tris60, v.index);
    const f3 em = tri.emissive();
    if (has_emission(em))
    {
        accum[px.idx] = {em.x, em.y, em.z, 1.0f};
        return ray;
    }
    const Surf surf = surface_from_visibility(tri, v.u, v.v, eye);
    const Res r = res.load(px.idx);
    if (shade)
    {
        shade->bg = (kInvPi * tri.color()) * geometry_term(surf.p, surf.n, r.s.hp, r.s.hn);
        shade->rad = r.s.rad;
        shade->ucw = r.ucw;
        return visibility_ray(surf.p, surf.n, r.s.hp);
    }
    write_accum(accum, px.idx, resolve_radiance(bvh, surf, tri.color(), r), opt.accumulate);
    return ray;
}

// ---- 07_pt.cu:11-90 (EX = 7), 08_nee.cu:11-129 (EX = 8), 09_ris.cu:11-166 (EX = 9)
// Returns the rays this pixel traced: closest-hit (camera + bounce rays) in the low 16 bits, shadow rays in the high 16
// (SURVEY.md section 8d: 08_nee 1 + 1 per path vertex; 09_ris 1 + 1, or 1 + 32 + 1 + 1 with the shadowed target function).
// LS: the light source, see k_pt_vertex (kernels_paths.cu)
template <int EX, class M, class LS = LightsIndexed>
CRT_HD uint32_t px_path_trace(const Pix& px, int W, int H, int frame, const Bvh& bvh, const float* tris60,
                              const typename LS::Elem* lights, uint32_t n_lights, const crt_raygen& raygen, const Opt& opt,
                              crt_float4* accum)
{
    uint32_t n_closest = 0, n_shadow = 0;
    Pcg rng(hash_pcg3(px.xi, px.yi, frame), 0);
    f3 ro, rd;
    primary_ray(raygen, px, W, H, ro, rd);
    f3 radiance = {0.0f, 0.0f, 0.0f}, throughput = {1.0f, 1.0f, 1.0f};
    for (int depth = 0; depth < opt.max_depth; ++depth)
    {
        Hit h;
        ++n_closest;
        if (!trace<false>(bvh, ro, rd, 0.0f, kFltMax, h))
        {
            if (EX == 7) radiance = radiance + throughput * opt.sky;
            break;
        }
        const TriRef tri = tri_at(tris60, h.prim);
        const f3 em = tri.emissive();
        if (has_emission(em))
        {
            if (EX == 7 || depth == 0) radiance = radiance + throughput * em;
            break;
        }
        const Surf surf = surface_from_hit(tri, ro, rd, h.t);
        const f3 color = tri.color();
        if (EX == 8)
        {
            const float r0 = rng.next_f();
            const float r1 = rng.next_f();
            const float r2 = rng.next_f();
            const LightSample ls = LS::at(tris60, lights, n_lights).sample(r0, r1, r2);
            ++n_shadow;
            const float V = check_visibility(bvh, surf.p, surf.n, ls.p);
            const f3 brdf = kInvPi * color;
            const float G = geometry_term(surf.p, surf.n, ls.p, ls.n);
            const float light_pdf = light_pdf_of<LS>(ls, n_lights);
            radiance = radiance + throughput * brdf * G * V * ls.emissive / light_pdf;
        }
        else if (EX == 9)
        {
            const Res r = ris_candidates(bvh, LS::at(tris60, lights, n_lights), surf, opt.ris_count, opt.shadowed, rng);
            n_shadow += 1u + (opt.shadowed ? (uint32_t)(opt.ris_count > 0 ? opt.ris_count : 0) + 1u : 0u);
            const f3 brdf = kInvPi * color;
            const float G = geometry_term(surf.p, surf.n, r.s.hp, r.s.hn);
            const float V = check_visibility(bvh, surf.p, surf.n, r.s.hp);
            const float p_hat = target_function(bvh, surf.p, surf.n, r.s.hp, r.s.hn, r.s.rad, opt.shadowed);
            radiance = radiance + throughput * brdf * G * V * r.s.rad * ucw_of(r, p_hat);
        }
        const f3 wo = bounce_direction<M>(surf, tri, rng);
        throughput = throughput * color;
        ro = surf.p + 0.001f * surf.n;  // offset_ray_position, core.hpp:32-36
        rd = wo;
    }
    write_accum(accum, px.idx, radiance, opt.accumulate);
    return n_closest | (n_shadow << 16);
}

// ---- 06_ao_hiprt.cu:35-91, N_Rays as a parameter; returns the RGBA8 pixel
template <class M>
CRT_HD uint32_t px_ao(const Pix& px, const crt_raygen& raygen, int W, int H, const Bvh& bvh, const float* tris60,
                      int n_rays, uint32_t& ao_rays_traced)
{
    ao_rays_traced = 0;
    Pcg rng(0, hash_pcg3(px.xi, px.yi, 42));
    f3 ro, rd;
    primary_ray(raygen, px, W, H, ro, rd);
    Hit h;
    if (!trace<false>(bvh, ro, rd, 0.0f, kFltMax, h)) return 32u | (32u << 8) | (32u << 16) | (255u << 24);
    const TriRef tri = tri_at(tris60, h.prim);
    const f3 v0 = tri.v(0), v1 = tri.v(1), v2 = tri.v(2);
    f3 n = tri_normal(v0, v1, v2);
    if (0.0f < dot(n, rd)) n = -n;
    const f3 t0 = normalize(v1 - v0);
    const f3 t1 = cross(t0, n);
    const f3 ao_ro = ro + rd * h.t + n * 0.0001f;
    int n_visible = 0;
    ao_rays_traced = (uint32_t)(n_rays > 0 ? n_rays : 0);
#if !defined(CRT_RAYS_PER_LANE)
    // the reference's loop shape: all lanes trace their i-th ray together (the per-lane loop below is slower, see RayLoop)
    for (int i = 0; i < n_rays; i++)
    {
        const float r0 = rng.next_f();
        const float r1 = rng.next_f();
        const float r2 = rng.next_f();
        const f3 s = sample_hemisphere<M>(r0, r1, r2);
        const f3 ao_rd = t0 * s.x + t1 * s.z + n * s.y;
        Hit ah;
        if (!trace<true>(bvh, ao_ro, ao_rd, 0.0f, kFltMax, ah)) n_visible++;
    }
#else
    // The n_rays walks of a pixel as one loop over walk steps: a lane whose ray is decided draws its next ray at once
    // instead of waiting for the warp's longest walk of the same ray index (the reference's `for` over rays traced in
    // lockstep ran at a third of the lanes: bench --config 06, profiles/r2/tuning.txt).  Per lane the rays, their random
    // numbers and their outcomes are the same sequence as before, so the pixel is too.
    int i = 0;
    bool walking = false;
    RaySetup r;
    Walk w;
    WalkStack stack;
    Hit ah;
    const RayLoop loop;
    for (;;)
    {
        bool start;
        if (!loop.next(!walking && i < n_rays, walking, start)) break;
        if (start && !walking && i < n_rays)
        {
            const float r0 = rng.next_f();
            const float r1 = rng.next_f();
            const float r2 = rng.next_f();
            const f3 s = sample_hemisphere<M>(r0, r1, r2);
            const f3 ao_rd = t0 * s.x + t1 * s.z + n * s.y;
            // the reference asks for the closest hit with maxT = FLT_MAX and only uses hit / no hit (:78-82)
            r = setup_ray(ao_ro, ao_rd);
            walk_begin(w, r);
            ah.prim = -1;
            ah.t = kFltMax;
            ah.u = ah.v = 0.0f;
            walking = true;
        }
        if (walking)
        {
            const int state = walk_step<true, true>(bvh, w, stack, r, 0.0f, ah, CRT_LANES_WALKING());
            if (state != kWalkContinue)
            {
                if (state == kWalkDone) n_visible++;
                i++;
                walking = false;
            }
        }
    }
#endif
    const float ao = (float)n_visible / (float)n_rays;
    const uint32_t c = (uint32_t)(M::pow(ao, 1.0f / 2.2f) * 255.0f) & 0xffu;
    return c | (c << 8) | (c << 16) | (255u << 24);
}
}  // namespace crt
