// TEST INFRASTRUCTURE — host build of the device functions of presampled light tiles (csrc/restir_core.cuh:
// light_tile_slot .. pixel_lights): the tile build in the order of csrc/geometry.cu: build_light_tiles, and the candidate
// bodies px_generate_candidate / px_candidate_temporal over LightsTiles, on tests/reuse/emu_reuse.cpp (the harness and the
// reuse modes) and tests/lights/emu_lights.cpp (the power table), both included unchanged, so that `pytest -m "not gpu"`
// checks the CUDA path's arithmetic against the CPU specification (tests/lights/tile_port.cpp).
#include "../reuse/emu_reuse.cpp"
#include "emu_lights.cpp"

namespace
{
// k_candidate_temporal[_reprojected] over any light source + k_trace_shadow_queue<2>, rays traced inline
template <class M, int RW, class L>
void candidate_temporal_any(int W, int H, int frame, const Bvh& bvh, const float* t60, const crt_visibility* vis, f3 eye,
                            const L& lights, const Opt& opt, const SoaStore& T, const GBuf& g, const Reprojection* rp)
{
    launch(W, H, [&](Pix p)
           {
               const CandPixel cp = classify_pixel(p, t60, vis);
               const DeferredRay d = rp ? px_candidate_temporal<M, L, true, RW>(p, cp, frame, bvh, t60, eye, lights, opt, T, g, HaloPeers(), 0u, *rp)
                                        : px_candidate_temporal<M, L, false, RW>(p, cp, frame, bvh, t60, eye, lights, opt, T, g);
               Hit h;
               if (d.want && !trace<true, true>(bvh, d.org, d.dir, 0.0f, 0.99f, h)) *T.mword(p.idx) |= kVisBit;
           });
}
}  // namespace

extern "C"
{
    // the uniform source records (k_build_light_table)
    void emu_uniform_table(const float* tris60, const uint32_t* lights, int nlights, float* out)
    {
        for (int i = 0; i < nlights; i++)
        {
            const LightRec r = make_light_rec(tris60, lights[i], (uint32_t)nlights);
            memcpy(out + 16 * (size_t)i, &r, sizeof r);
        }
    }
    // k_light_tiles: T * S records of `frame` from K source records
    void emu_light_tiles(const float* src, uint32_t K, int frame, int log2_t, int log2_s, float* out)
    {
        const uint32_t count = 1u << (log2_t + log2_s);
        for (uint32_t i = 0; i < count; i++)
            memcpy(out + 16 * (size_t)i, src + 16 * (size_t)light_tile_slot((uint32_t)frame, i >> log2_s, i & ((1u << log2_s) - 1u), K),
                   64);
    }
    // k_generate_candidate<LightsTiles, ...> without shadowed target function (tiles: this frame's records)
    void emu_generate_candidate_tiles(int W, int H, int frame, void* gp, const crt_triangle* tris, const crt_visibility* vis,
                                      const float* eye, const float* tiles, int log2_t, int log2_s, const crt_options* opt,
                                      crt_reservoir* res)
    {
        const Bvh bvh = ((EmuGeom*)gp)->view();
        const LightsTiles L{(const LightRec*)tiles, (uint32_t)log2_t, (uint32_t)log2_s};
        launch(W, H, [&](Pix p) { px_generate_candidate(p, frame, bvh, (const float*)tris, vis, v3(eye), L, make_opt(*opt), AosStore{res}); });
    }
    // the fused frame (rw_restir_frame_fast[_reprojected]'s kernel sequence) with the candidates drawn from `tiles`;
    // prev_rg != nullptr with temporal reuse: k_candidate_temporal_reprojected
    void emu_restir_frame_fast_tiles(int W, int H, int frame, void* gp, const crt_triangle* tris, const crt_raygen* rg,
                                     const float* eye_p, const float* tiles, int log2_t, int log2_s, const crt_options* options,
                                     crt_visibility* vis, char* temporal, char* res_a, char* res_b, crt_float4* accum,
                                     uint32_t* pixels, const crt_raygen* prev_rg, const crt_visibility* prev_vis)
    {
        const Bvh bvh = ((EmuGeom*)gp)->view();
        const float* t60 = (const float*)tris;
        const f3 eye = v3(eye_p);
        const Opt opt = make_opt(*options);
        const size_t n = (size_t)W * H;
        std::vector<char> g0(n * 16), g1(n * 8);
        std::vector<uint8_t> cls(n, 0);
        const GBuf g{g0.data(), g1.data(), cls.data()};
        const SoaStore T{temporal, n}, A{res_a, n}, B{res_b, n};
        const LightsTiles L{(const LightRec*)tiles, (uint32_t)log2_t, (uint32_t)log2_s};
        launch(W, H, [&](Pix p) { px_raycast(p, W, H, bvh, *rg, vis); });
        std::vector<char> snapshot(temporal, temporal + n * 72);
        Reprojection rp;
        const bool reproject = prev_rg && options->use_temporal_resampling;
        if (reproject)
        {
            rp.history = SoaStore{snapshot.data(), n};
            rp.prev_cam = *prev_rg;
            rp.W = W;
            rp.H = H;
            rp.prev_vis = prev_vis;
            rp.prev_eye = f3{prev_rg->m_origin.x, prev_rg->m_origin.y, prev_rg->m_origin.z};
        }
        const Reprojection* rpp = reproject ? &rp : nullptr;
        RW_CALL(candidate_temporal_any, W, H, frame, bvh, t60, vis, eye, L, opt, T, g, rpp);
        SoaStore in = T, out = A;
        if (opt.spatial)
            for (int pass = 0; pass < options->spatial_resampling_passes; pass++)
            {
                if (pass == 1) { in = A; out = B; }
                else if (pass > 1) std::swap(in, out);
                RW_CALL(spatial_fast_all, W, H, frame, pass, bvh, eye, opt, in, out, g);
            }
        const SoaStore fin = opt.spatial && options->spatial_resampling_passes > 0 ? out : T;
        launch(W, H, [&](Pix p)
               {
                   DeferredShade sh{{0, 0, 0}, {0, 0, 0}, 0.0f};
                   const DeferredRay d = px_resolve_fast(p, accum, t60, vis, fin, g, sh, opt.accumulate, opt.reuse);
                   if (!d.want) return;
                   Hit h;
                   const float V = trace<true>(bvh, d.org, d.dir, 0.0f, 0.99f, h) ? 0.0f : 1.0f;
                   write_accum(accum, p.idx, sh.bg * V * sh.rad * sh.ucw, opt.accumulate);  // shadow_epilogue<kEpiResolve>
               });
        orc_tone_mapping(pixels, accum, W, H);
    }
}
