// restir_fast.cuh — per-pixel bodies of the fused frame ("fast mode", crt_restir_di_frame):
// the same arithmetic as restir_pixel.cuh, in the same order, on a different data flow.
//
//   * reservoirs live in sector-planar form inside the TypedBuffer<Reservoir> allocations (SoaStore below): two
//     32-byte planes and one 8-byte plane, 72 B/px, every access a 256-bit (64-bit) load or store, a warp's 8x4
//     pixel tile touching full 128-byte lines;
//   * generate_candidate + temporal_resampling are one body: the candidate reservoir stays in registers, the
//     merged reservoir is written in place over last frame's (same pixel: no reprojection in the reference,
//     10_restir_di.cu:178), which also makes save_temporal_reservoir (:239-254) a no-op;
//   * the visibility-reuse ray (:127-131) is only emitted when this frame's candidate survives the temporal
//     merge — otherwise Reservoir::merge (reservoir.hpp:31-37) overwrites the sample, visibility included, and
//     the reference's traced value is never read;
//   * the surface point/normal the reference rebuilds from Visibility + Triangle in every kernel
//     (make_surface_info, core.hpp:188-207) is computed once and kept in a small G-buffer together with a
//     1-byte pixel class; the spatial pass rejects sky/emissive neighbours (:317-326) from a marker bit inside
//     the neighbour's own reservoir record, so the rejection costs no gather of its own;
//   * tone mapping (common.cu:30-74) stays a separate sweep: inside the ray tracer's epilogue its three powf calls
//     ran once per finished ray with a handful of live lanes and cost 1.0 ms per 4K frame (profiles/r1, state h)
//     against 0.1 ms as a kernel of its own.
//
// Host-callable like restir_pixel.cuh, so tests/emu runs these bodies on the CPU against the oracle.
#pragma once
#include "restir_pixel.cuh"

namespace crt
{
struct u2 { uint32_t x, y; };
CRT_HD void store_u4(void* p, u4 v)
{
#if defined(__CUDA_ARCH__)
    *(uint4*)p = make_uint4(v.x, v.y, v.z, v.w);
#else
    memcpy(p, &v, 16);
#endif
}
CRT_HD u2 load_u2(const void* p)
{
#if defined(__CUDA_ARCH__)
    const uint2 v = __ldg((const uint2*)p);
    return {v.x, v.y};
#else
    u2 v;
    memcpy(&v, p, 8);
    return v;
#endif
}
CRT_HD void store_u2(void* p, u2 v)
{
#if defined(__CUDA_ARCH__)
    *(uint2*)p = make_uint2(v.x, v.y);
#else
    memcpy(p, &v, 8);
#endif
}

// Sector-planar reservoir storage over n pixels (n * 72 bytes used of the n * 76 the reference allocates).
// The unit of a random gather is the 32-byte sector, and the L1 charges one wavefront per distinct line per load
// instruction, so the fields are grouped by *who reads them together*, one 256-bit load per group:
//   plane 0 @ 0      32 B/px  origin_position.xyz, origin_normal.xyz, flags | M, ucw
//   plane 1 @ 32 n   32 B/px  hit_position.xyz, hit_normal.xyz, radiance.x, radiance.y
//   plane 2 @ 64 n    8 B/px  radiance.z, w_sum
// Plane 0 alone answers everything the spatial pass asks of a neighbour whose sample is occluded (visibility reuse:
// p_hat * 0 — its weight is +0 whatever the sample is, only M after the rejection heuristics and one random number
// are consumed) and tells sky/emissive pixels apart (kSkipBit), so most neighbours cost one sector instead of the
// six (five planes + the class byte) of the earlier 16-byte planes (profiles/r1: k_spatial_fast at 71 % of the L1's
// wavefront rate with 18 % of DRAM bandwidth).  Planes 1 and 2 are fetched for visible neighbours only.
//   flags | M word:  bit 31 sample.visibility    bit 30 kTracedBit    bit 29 kSkipBit    bits 0..28 M
// kTracedBit: the visibility bit is the outcome of check_visibility(origin_position, origin_normal, hit_position)
// traced by this library against the current geometry (k_trace_shadow_queue<2>); it travels with the sample through
// merges.  resolve uses it: when the final sample's origin is bit for bit this pixel's surface, the shadow ray of
// 10_restir_di.cu:443-444 is the ray already traced, and its stored answer is used instead of tracing it again.
constexpr int kSoaPlanes = 3;
constexpr int kHaloRows = 87;  // rows a spatial pass can reach beyond a slab at the reference's radius 30: |offset| <= 86.4 px (10_restir_di.cu:309-313)
// the same bound for any radius: offset = radius / 1.96 * sqrt(-2 ln rv0) * cos|sin, rv0 >= 2^-23, truncated towards
// zero — which rounds the reach up on the side of smaller coordinates: floor(offset) + 1 rows; the factor covers the
// float rounding of the product (python/slabs.py: halo_rows is the same formula)
inline int halo_rows_for(float radius)
{
    return (int)floor(fabs((double)radius) / 1.96 * sqrt(-2.0 * log(ldexp(1.0, -23))) * (1.0 + 1e-5)) + 1;
}
CRT_HD size_t soa_plane_offset(int plane, size_t n) { return (size_t)plane * 32u * n; }
CRT_HD size_t soa_plane_elem(int plane) { return plane < 2 ? 32u : 8u; }
constexpr uint32_t kVisBit = 0x80000000u, kTracedBit = 0x40000000u, kSkipBit = 0x20000000u, kMMask = 0x1fffffffu;
constexpr uint32_t kSampleVisible = 1u, kSampleTraced = 2u;  // Sample::vis in registers
constexpr int kMWord = 6;                                    // word of the plane-0 record holding flags | M

CRT_HD void store_u8w(void* p, const u8w& v)
{
#if defined(__CUDA_ARCH__)
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v.lo.x), "r"(v.lo.y), "r"(v.lo.z),
                 "r"(v.lo.w), "r"(v.hi.x), "r"(v.hi.y), "r"(v.hi.z), "r"(v.hi.w)
                 : "memory");
#else
    memcpy(p, &v, 32);
#endif
}
CRT_HD bool same_bits(f3 a, f3 b) { return f2u(a.x) == f2u(b.x) && f2u(a.y) == f2u(b.y) && f2u(a.z) == f2u(b.z); }

// plane 0 of one reservoir: what a neighbour merge needs before it knows whether the sample can be selected at all
struct ResHead
{
    f3 op, on;
    uint32_t mword;
    float ucw;
    CRT_HD bool skip() const { return (mword & kSkipBit) != 0u; }
    CRT_HD bool visible() const { return (mword & kVisBit) != 0u; }
    CRT_HD int M() const { return (int)(mword & kMMask); }
};

struct SoaStore
{
    char* base;
    size_t n;
    CRT_HD char* plane(int p, int idx) const { return base + soa_plane_offset(p, n) + (size_t)idx * soa_plane_elem(p); }
    CRT_HD ResHead load_head(int idx) const
    {
        const u8w a = load_u8w(plane(0, idx));
        return ResHead{{u2f(a.lo.x), u2f(a.lo.y), u2f(a.lo.z)}, {u2f(a.lo.w), u2f(a.hi.x), u2f(a.hi.y)}, a.hi.z, u2f(a.hi.w)};
    }
    // the rest of a reservoir whose head has been read; a skipped pixel reads as Reservoir{} whatever planes 1-2 hold
    CRT_HD Res finish_load(int idx, const ResHead& h) const
    {
        if (h.skip()) return empty_res();
        const u8w b = load_u8w(plane(1, idx));
        const u2 c = load_u2(plane(2, idx));
        Res r;
        r.s.op = h.op;
        r.s.on = h.on;
        r.s.hp = {u2f(b.lo.x), u2f(b.lo.y), u2f(b.lo.z)};
        r.s.hn = {u2f(b.lo.w), u2f(b.hi.x), u2f(b.hi.y)};
        r.s.rad = {u2f(b.hi.z), u2f(b.hi.w), u2f(c.x)};
        r.s.vis = (h.mword >> 31) | ((h.mword & kTracedBit) ? kSampleTraced : 0u);
        r.w_sum = u2f(c.y);
        r.ucw = h.ucw;
        r.M = h.M();
        return r;
    }
    CRT_HD Res load(int idx) const { return finish_load(idx, load_head(idx)); }
    CRT_HD void store(int idx, const Res& r) const
    {
        const uint32_t mword = ((uint32_t)r.M & kMMask) | ((r.s.vis & kSampleVisible) ? kVisBit : 0u) |
                               ((r.s.vis & kSampleTraced) ? kTracedBit : 0u);
        store_u8w(plane(0, idx), u8w{{f2u(r.s.op.x), f2u(r.s.op.y), f2u(r.s.op.z), f2u(r.s.on.x)},
                                     {f2u(r.s.on.y), f2u(r.s.on.z), mword, f2u(r.ucw)}});
        store_u8w(plane(1, idx), u8w{{f2u(r.s.hp.x), f2u(r.s.hp.y), f2u(r.s.hp.z), f2u(r.s.hn.x)},
                                     {f2u(r.s.hn.y), f2u(r.s.hn.z), f2u(r.s.rad.x), f2u(r.s.rad.y)}});
        store_u2(plane(2, idx), u2{f2u(r.s.rad.z), f2u(r.w_sum)});
    }
    // a sky / emissive pixel: Reservoir{} with the class marker; planes 1-2 are not touched (never read for it)
    CRT_HD void store_skip(int idx) const { store_u8w(plane(0, idx), u8w{{0u, 0u, 0u, 0u}, {0u, 0u, kSkipBit, 0u}}); }
    // word holding flags | M (the shadow-ray kernel sets kVisBit for unoccluded candidates)
    CRT_HD uint32_t* mword(int idx) const { return (uint32_t*)plane(0, idx) + kMWord; }
};

// G-buffer of the fused frame: surface point and shading normal of the primary hit, and the pixel class
enum : uint8_t { kPixSkip = 0, kPixDiffuse = 1 };  // skip = sky or emissive: no reservoir work (10_restir_di.cu:62-70)
struct GBuf
{
    char* g0;      // float4 per pixel: p.xyz, n.x
    char* g1;      // float2 per pixel: n.y, n.z
    uint8_t* cls;  // kPix*
    CRT_HD Surf load(int idx) const
    {
        const u4 a = load_u4(g0 + (size_t)idx * 16);
        const u2 b = load_u2(g1 + (size_t)idx * 8);
        return Surf{{u2f(a.x), u2f(a.y), u2f(a.z)}, {u2f(a.w), u2f(b.x), u2f(b.y)}};
    }
    CRT_HD void store(int idx, const Surf& s) const
    {
        store_u4(g0 + (size_t)idx * 16, u4{f2u(s.p.x), f2u(s.p.y), f2u(s.p.z), f2u(s.n.x)});
        store_u2(g1 + (size_t)idx * 8, u2{f2u(s.n.y), f2u(s.n.z)});
    }
    CRT_HD uint8_t pixel_class(int idx) const
    {
#if defined(__CUDA_ARCH__)
        return __ldg(cls + idx);
#else
        return cls[idx];
#endif
    }
};

// Multi-GPU row slabs (slab_p2p.cu): the neighbouring slabs' copies of the buffer a kernel writes.  A pixel whose
// row lies within kHaloRows of the slab boundary is stored there too — the halo rows travel over NVLink from the
// producing kernel's own epilogue, overlapped with the rest of the kernel, instead of in a copy afterwards.
struct HaloPeers
{
    char* up = nullptr;         // reservoir storage of the slab above (rows yi < up_end are mirrored there)
    char* down = nullptr;       // ... of the slab below (rows yi >= down_begin)
    uint8_t* up_cls = nullptr;  // pixel-class planes (candidate kernel only)
    uint8_t* down_cls = nullptr;
    int up_end = 0, down_begin = 0;
    CRT_HD void mirror(const Pix& px, size_t n, const Res& r) const
    {
        if (up && px.yi < up_end) SoaStore{up, n}.store(px.idx, r);
        if (down && px.yi >= down_begin) SoaStore{down, n}.store(px.idx, r);
    }
    CRT_HD void mirror_skip(const Pix& px, size_t n) const
    {
        if (up && px.yi < up_end) SoaStore{up, n}.store_skip(px.idx);
        if (down && px.yi >= down_begin) SoaStore{down, n}.store_skip(px.idx);
    }
    CRT_HD void mirror_class(const Pix& px, uint8_t c) const
    {
        if (up_cls && px.yi < up_end) up_cls[px.idx] = c;
        if (down_cls && px.yi >= down_begin) down_cls[px.idx] = c;
    }
};

// ---- generate_candidate (10_restir_di.cu:36-135) + temporal_resampling (:137-237) + save (:239-254).
// `temporal` holds last frame's post-temporal reservoirs on entry and this frame's on exit.
// Requires !opt.shadowed (the fused frame falls back to the per-kernel path otherwise).
// Returns the visibility-reuse ray if one has to be traced; the reservoir is then stored with
// visibility = false and the tracer sets the bit for an unoccluded ray.
// The pixel's class is decided first and on its own (classify_pixel) so that a kernel can ballot the diffuse lanes
// of a warp at a point every lane reaches, and hand the loop the mask of complete lane pairs (LightsTable::fetch).
struct CandPixel
{
    Vis v;
    bool skip;  // sky or emissive: no reservoir work (10_restir_di.cu:52-70)
};
CRT_HD CandPixel classify_pixel(const Pix& px, const float* tris60, const crt_visibility* vis)
{
    CandPixel c{load_vis(vis, px.idx), false};
    c.skip = c.v.index == -1 || has_emission(tri_at(tris60, c.v.index).emissive());
    return c;
}
// lanes of `lanes` whose pair partner (lane ^ 1) is in `lanes` too
CRT_HD unsigned complete_pairs(unsigned lanes) { return lanes & (((lanes & 0x55555555u) << 1) | ((lanes & 0xaaaaaaaau) >> 1)); }

// REPROJ (extension, DESIGN.md section 11): the history is read from `history` — a snapshot of last frame's `temporal` —
// at the pixel this surface point had in the previous frame's camera (reproject_pixel, restir_core.cuh), Reservoir{} when
// it had none; `temporal` is only written.  Otherwise the history is `temporal` at this pixel, merged in place.
// prev_vis / prev_eye: the previous frame's Visibility buffer and eye (crt_restir_set_previous_frame), read by
// CRT_REUSE_UNBIASED only — the history pixel's surface (DESIGN.md section 15)
struct Reprojection
{
    SoaStore history{nullptr, 0};
    crt_raygen prev_cam{};
    int W = 0, H = 0;
    const crt_visibility* prev_vis = nullptr;
    f3 prev_eye{0.0f, 0.0f, 0.0f};
};
// RW: CRT_REUSE_REFERENCE, or CRT_REUSE_UNBIASED: temporal_merge_unbiased, and with REPROJ
// temporal_merge_unbiased_reprojected on the history pixel's previous surface — one 16-byte Visibility load and the
// triangle's 36 vertex bytes at the history pixel, only when the history has M > 0
// MOTION (with REPROJ; crt_restir_set_previous_triangles): `prev_tris60` is the previous frame's triangle array; the
// look-up and the history's surface follow moved triangles as px_temporal<..., MOTION> does (DESIGN.md section 17)
template <class M, class L, bool REPROJ = false, int RW = CRT_REUSE_REFERENCE, bool MOTION = false>
CRT_HD DeferredRay px_candidate_temporal(const Pix& px, const CandPixel& cp, int frame, const Bvh& bvh, const float* tris60,
                                         f3 eye, const L& lights, const Opt& opt_in, const SoaStore& temporal,
                                         const GBuf& g, const HaloPeers& peers = HaloPeers(), unsigned pair_mask = 0u,
                                         const Reprojection& rp = Reprojection(), const float* prev_tris60 = nullptr)
{
    Opt opt = opt_in;
    opt.shadowed = false;  // compile-time constant here: no traversal code inside the target function
    DeferredRay ray{false, {0, 0, 0}, {0, 0, 0}};
    const Vis v = cp.v;
    if (cp.skip)
    {
        g.cls[px.idx] = kPixSkip;
        peers.mirror_class(px, kPixSkip);
        temporal.store_skip(px.idx);  // reads back as what the reference leaves there: Reservoir{} copied by save_temporal
        peers.mirror_skip(px, temporal.n);
        return ray;
    }
    const TriRef tri = tri_at(tris60, v.index);
    g.cls[px.idx] = kPixDiffuse;
    peers.mirror_class(px, kPixDiffuse);
    Pcg rng(hash_pcg4(px.xi, px.yi, frame, 0), 0);
    const Surf surf = surface_from_visibility(tri, v.u, v.v, eye);
    g.store(px.idx, surf);
    Res r = ris_candidates(bvh, pixel_lights(lights, px.xi, px.yi, frame), surf, opt.ris_count, false, rng, pair_mask);
    r.ucw = ucw_of(r, target_function(bvh, surf.p, surf.n, r.s.hp, r.s.hn, r.s.rad, false));
    bool candidate_survives = true;
    if (opt.temporal)
    {
        Pcg rng_t(hash_pcg4(px.xi, px.yi, frame, 1), 0);
        Res history;
        bool has_h = false;
        Surf hsurf{};
        if (REPROJ)
        {
            int xp, yp;
            const f3 p_prev = MOTION ? previous_point(tris60, prev_tris60, v, surf) : surf.p;
            const bool found = reproject_pixel(to_raygen(rp.prev_cam), rp.W, rp.H, p_prev, xp, yp);
            history = found ? rp.history.load(xp + (rp.H - yp - 1) * rp.W) : empty_res();
            if (RW == CRT_REUSE_UNBIASED && found && history.M > 0)
                has_h = previous_surface<MOTION>(rp.prev_vis, tris60, xp + (rp.H - yp - 1) * rp.W, rp.prev_eye, hsurf,
                                                 prev_tris60);
        }
        else history = temporal.load(px.idx);
        if (RW == CRT_REUSE_UNBIASED && REPROJ)
            candidate_survives = !temporal_merge_unbiased_reprojected<M>(bvh, surf, has_h, hsurf, eye, opt, history, r, rng_t);
        else if (RW == CRT_REUSE_UNBIASED) candidate_survives = !temporal_merge_unbiased<M>(bvh, surf, eye, opt, history, r, rng_t);
        else candidate_survives = !temporal_merge<M>(bvh, surf, eye, opt, history, r, rng_t);
    }
    if (opt.reuse && candidate_survives)
    {
        // a ray that its own triangle stops (a candidate below the surface's horizon: 31 % of them) is decided here
        ray = visibility_ray_past_own(surf.p, surf.n, r.s.hp, tri);
        r.s.vis = kSampleTraced;  // visibility = false until the tracer finds the ray unoccluded
    }
    temporal.store(px.idx, r);
    peers.mirror(px, temporal.n, r);  // visibility still pending for a deferred ray: the tracer mirrors the final word
    return ray;
}

// The G-buffer record of a pixel outside this context's row range (crt_restir_set_halo_surfaces): what px_candidate_temporal
// stores there on the context that owns the row — the same Visibility record (the same primary ray, traced into a buffer of
// this context's own), the same surface_from_visibility with this frame's eye.  Sky and emissive pixels get no record (the
// spatial pass skips them by the neighbour's kSkipBit before it reads one), and the class plane is not written: with slab
// links the neighbours store into those rows of it.
CRT_HD void px_halo_surface(const Pix& px, const float* tris60, const crt_visibility* vis, f3 eye, const GBuf& g)
{
    const CandPixel cp = classify_pixel(px, tris60, vis);
    if (cp.skip) return;
    g.store(px.idx, surface_from_visibility(tri_at(tris60, cp.v.index), cp.v.u, cp.v.v, eye));
}

// px_spatial's unbiased form (CRT_REUSE_UNBIASED) on this data flow, from the pixel's input reservoir `r` and its random
// stream: a neighbour's surface is its G-buffer record (24 bytes) instead of plane 0's sample origin, planes 1-2 are read
// for every visited neighbour (the visibility bit weighs nothing, so there is no weightless shortcut), and the replayed
// second pass sums Z.  The G-buffer must hold every neighbour's row: the whole image on one context, or the halo rows
// px_halo_surface fills on a row range.
template <class M>
CRT_HD void spatial_fast_unbiased(const Pix& px, int W, int H, const Bvh& bvh, f3 eye, const Opt& opt, const SoaStore& in,
                                  const GBuf& g, const Surf& surf, Pcg rng, Res& r)
{
    const Pcg rng_z = rng;
    const int c_own = r.M;
    for (int k = 0; k < opt.spatial_count; ++k)
    {
        int x, y;
        spatial_neighbour<M>(px.xi, px.yi, opt.radius, rng, x, y);
        if (x < 0 || x >= W || y < 0 || y >= H) continue;
        if (x == px.xi && y == px.yi) continue;
        const int pid = x + (H - y - 1) * W;
        const ResHead nh = in.load_head(pid);
        if (nh.skip()) continue;
        const int c = confidence<M>(nh.M(), surf, g.load(pid), eye);
        const float u = rng.next_f();
        const Res nb = in.finish_load(pid, nh);
        const float weight = target_function(bvh, surf.p, surf.n, nb.s.hp, nb.s.hn, nb.s.rad, false) * nb.ucw * (float)c;
        r.w_sum += weight;  // spatial_merge_unbiased
        r.M += c;
        if (u < weight / r.w_sum) r.s = nb.s;
    }
    const float p_hat = target_function(bvh, surf.p, surf.n, r.s.hp, r.s.hn, r.s.rad, false);
    int z = c_own;
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
            const ResHead nh = in.load_head(pid);
            if (nh.skip()) continue;
            const Surf ns = g.load(pid);
            (void)rz.next_f();  // the merge's random number
            z = z_of(z, confidence<M>(nh.M(), surf, ns, eye), bvh, ns, r.s, false);
        }
    }
    r.ucw = ucw_unbiased(r.w_sum, z, p_hat);
}

// ---- spatial_resampling (10_restir_di.cu:256-388) with opt.spatial == true (the disabled form is a copy the
// fused frame skips).
// A neighbour whose sample is occluded (visibility reuse, :352-355: p_hat_y *= visibility) merges with weight
// p_hat_y * 0 * ucw * M = +0: w_sum and the sample stay as they are, M grows by the neighbour's M after the
// rejection heuristics and one random number is drawn.  That needs plane 0 of the neighbour only.  (Precondition,
// true for every finite scene: the target function of the neighbour's sample is finite — it is not only if the
// light sample coincides bit for bit with this pixel's surface point — and ucw is finite, which is checked.)
// RW = CRT_REUSE_UNBIASED: spatial_fast_unbiased above
template <class M, int RW = CRT_REUSE_REFERENCE>
CRT_HD void px_spatial_fast(const Pix& px, int W, int H, int frame, int pass, const Bvh& bvh, f3 eye, const Opt& opt_in,
                            const SoaStore& in, const SoaStore& out, const GBuf& g, const HaloPeers& peers = HaloPeers())
{
    Opt opt = opt_in;
    opt.shadowed = false;
    if (g.pixel_class(px.idx) == kPixSkip)
    {
        // the reference leaves its output untouched; here the record carries the class marker the next pass's
        // neighbours (and the export) read
        out.store_skip(px.idx);
        peers.mirror_skip(px, out.n);
        return;
    }
    Pcg rng(hash_pcg4(px.xi, px.yi, frame, 2 + pass), 0);
    const Surf surf = g.load(px.idx);
    Res r = in.load(px.idx);
    if (RW == CRT_REUSE_UNBIASED) spatial_fast_unbiased<M>(px, W, H, bvh, eye, opt, in, g, surf, rng, r);
    else
    {
        for (int k = 0; k < opt.spatial_count; ++k)
        {
            int x, y;
            spatial_neighbour<M>(px.xi, px.yi, opt.radius, rng, x, y);
            if (x < 0 || x >= W || y < 0 || y >= H) continue;
            if (x == px.xi && y == px.yi) continue;
            const int pid = x + (H - y - 1) * W;
            const ResHead nh = in.load_head(pid);
            if (nh.skip()) continue;
            // common to every neighbour (the warp stays converged here): M after the rejection heuristics, one random
            Sample ns;
            ns.op = nh.op;
            ns.on = nh.on;
            const int nM = rejected_m<M>(r.s, ns, nh.M(), eye);
            const float u = rng.next_f();
            // only a neighbour that can be selected needs its sample: planes 1-2 and the target function
            float weight = 0.0f;
            Res nb;
            const bool weightless = opt.reuse && !nh.visible() && (f2u(nh.ucw) & 0x7f800000u) != 0x7f800000u;
            if (!weightless)
            {
                nb = in.finish_load(pid, nh);
                float p_hat_y = target_function(bvh, surf.p, surf.n, nb.s.hp, nb.s.hn, nb.s.rad, false);
                if (opt.reuse) p_hat_y *= (nb.s.vis & 1u) ? 1.0f : 0.0f;
                weight = p_hat_y * nb.ucw * (float)nM;
            }
            r.w_sum += weight;  // Reservoir::merge (reservoir.hpp:31-37)
            r.M += nM;
            if (!weightless && u < weight / r.w_sum) r.s = nb.s;
        }
        r.ucw = ucw_of(r, target_function(bvh, surf.p, surf.n, r.s.hp, r.s.hn, r.s.rad, false));
    }
    out.store(px.idx, r);
    peers.mirror(px, out.n, r);
}

// ---- resolve (10_restir_di.cu:390-459).  Sky/emissive pixels are finished here; for the others the shadow ray
// and the shading factors are returned (see px_resolve) — unless the ray has been traced already: a sample whose
// origin is bit for bit this pixel's surface and whose visibility carries kSampleTraced got that visibility from
// check_visibility(surf.p, surf.n, hit_position), the very call of :443-444, so the pixel is shaded here
// (`reuse_traced`; false reproduces the reference's ray count).
template <class RS>
CRT_HD DeferredRay px_resolve_fast(const Pix& px, crt_float4* accum, const float* tris60,
                                   const crt_visibility* vis, const RS& res, const GBuf& g, DeferredShade& shade,
                                   bool accumulate = true, bool reuse_traced = false)
{
    DeferredRay ray{false, {0, 0, 0}, {0, 0, 0}};
    const Vis v = load_vis(vis, px.idx);
    if (g.pixel_class(px.idx) == kPixSkip)
    {
        f3 c{0.0f, 0.0f, 0.0f};
        if (v.index != -1) c = tri_at(tris60, v.index).emissive();
        accum[px.idx] = {c.x, c.y, c.z, 1.0f};  // assigned even when accumulating
        return ray;
    }
    const Surf surf = g.load(px.idx);
    const Res r = res.load(px.idx);
    shade.bg = (kInvPi * tri_at(tris60, v.index).color()) * geometry_term(surf.p, surf.n, r.s.hp, r.s.hn);
    shade.rad = r.s.rad;
    shade.ucw = r.ucw;
    if (reuse_traced && (r.s.vis & kSampleTraced) && same_bits(r.s.op, surf.p) && same_bits(r.s.on, surf.n))
    {
        // radiance = brdf * G * V * sample.radiance * ucw, left to right (:446-447), as in shadow_epilogue
        const float V = (r.s.vis & kSampleVisible) ? 1.0f : 0.0f;
        write_accum(accum, px.idx, shade.bg * V * shade.rad * shade.ucw, accumulate);
        return ray;
    }
    return visibility_ray(surf.p, surf.n, r.s.hp);
}
// AoS <-> SoA conversion of one reservoir (crt_reservoir_export_aos / crt_reservoir_import_aos)
CRT_HD void soa_to_aos(const SoaStore& s, crt_reservoir* aos, int idx) { AosStore{aos}.store(idx, s.load(idx)); }
CRT_HD void aos_to_soa(const crt_reservoir* aos, const SoaStore& s, int idx)
{
    s.store(idx, AosStore{const_cast<crt_reservoir*>(aos)}.load(idx));
}
}  // namespace crt
