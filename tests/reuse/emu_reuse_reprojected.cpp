// TEST INFRASTRUCTURE — host build of the device bodies of the unbiased reuse weights with a moving camera
// (crt_temporal_resampling_reprojected_surfaces, crt_restir_set_previous_frame): tests/reuse/emu_reuse.cpp (included
// unchanged) plus px_temporal with a previous camera and the previous frame's Visibility, and the fused frame with
// px_candidate_temporal<..., REPROJ = true>, so that `pytest -m "not gpu"` checks them against the CPU specification
// (tests/reuse/reuse_port_reprojected.cpp).
#include "emu_reuse.cpp"

namespace
{
template <class M, int RW>
void temporal_reprojected_all(int W, int H, int frame, const Bvh& bvh, const float* t, const crt_visibility* vis, f3 eye,
                              const Opt& o, const crt_raygen* prev_cam, const crt_visibility* prev_vis, crt_reservoir* prev,
                              crt_reservoir* res)
{
    launch(W, H, [&](Pix p) { px_temporal<M, RW>(p, frame, bvh, t, vis, eye, o, AosStore{prev}, AosStore{res}, prev_cam, W, H, prev_vis); });
}
// k_candidate_temporal_reprojected + k_trace_shadow_queue<2>: the visibility-reuse rays traced inline
template <class M, int RW>
void candidate_temporal_reprojected_all(int W, int H, int frame, const Bvh& bvh, const float* t60, const crt_visibility* vis,
                                        f3 eye, const LightsIndexed& L, const Opt& opt, const SoaStore& T, const GBuf& g,
                                        const Reprojection& rp)
{
    launch(W, H, [&](Pix p)
           {
               const DeferredRay d = px_candidate_temporal<M, LightsIndexed, true, RW>(p, classify_pixel(p, t60, vis), frame, bvh,
                                                                                  t60, eye, L, opt, T, g, HaloPeers(), 0u, rp);
               Hit h;
               if (d.want && !trace<true, true>(bvh, d.org, d.dir, 0.0f, 0.99f, h)) *T.mword(p.idx) |= kVisBit;
           });
}
}  // namespace

extern "C"
{
    // px_temporal with a previous camera and the previous frame's Visibility (crt_temporal_resampling_reprojected_surfaces)
    void rw_temporal_resampling_reprojected(int W, int H, int frame, void* gp, const crt_triangle* tris, int,
                                            const crt_visibility* vis, const float* eye, const crt_options* opt,
                                            const crt_raygen* prev_cam, const crt_visibility* prev_vis,
                                            const crt_reservoir* prev, crt_reservoir* res)
    {
        RW_CALL(temporal_reprojected_all, W, H, frame, ((EmuGeom*)gp)->view(), (const float*)tris, vis, v3(eye),
                make_opt(*opt), prev_cam, prev_vis, (crt_reservoir*)prev, res);
    }

    // the fused frame with crt_restir_set_previous_frame: rw_restir_frame_fast's kernel sequence, the history read from a
    // snapshot of `temporal` at the reprojected pixel; prev_rg == nullptr (the first frame): rw_restir_frame_fast
    void rw_restir_frame_fast_reprojected(int W, int H, int frame, void* gp, const crt_triangle* tris, const crt_raygen* rg,
                                          const float* eye_p, const uint32_t* lights, int nlights, const crt_options* options,
                                          crt_visibility* vis, char* temporal, char* res_a, char* res_b, crt_float4* accum,
                                          uint32_t* pixels, const crt_raygen* prev_rg, const crt_visibility* prev_vis)
    {
        if (!prev_rg || !options->use_temporal_resampling)
        {
            rw_restir_frame_fast(W, H, frame, gp, tris, rg, eye_p, lights, nlights, options, vis, temporal, res_a, res_b, accum,
                                 pixels);
            return;
        }
        const Bvh bvh = ((EmuGeom*)gp)->view();
        const float* t60 = (const float*)tris;
        const f3 eye = v3(eye_p);
        const Opt opt = make_opt(*options);
        const size_t n = (size_t)W * H;
        std::vector<char> g0(n * 16), g1(n * 8);
        std::vector<uint8_t> cls(n, 0);
        const GBuf g{g0.data(), g1.data(), cls.data()};
        const SoaStore T{temporal, n}, A{res_a, n}, B{res_b, n};
        const LightsIndexed L{t60, lights, (uint32_t)nlights};
        launch(W, H, [&](Pix p) { px_raycast(p, W, H, bvh, *rg, vis); });
        std::vector<char> snapshot(temporal, temporal + n * 72);
        Reprojection rp;
        rp.history = SoaStore{snapshot.data(), n};
        rp.prev_cam = *prev_rg;
        rp.W = W;
        rp.H = H;
        rp.prev_vis = prev_vis;
        rp.prev_eye = f3{prev_rg->m_origin.x, prev_rg->m_origin.y, prev_rg->m_origin.z};
        RW_CALL(candidate_temporal_reprojected_all, W, H, frame, bvh, t60, vis, eye, L, opt, T, g, rp);
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
