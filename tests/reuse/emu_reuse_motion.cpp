// TEST INFRASTRUCTURE — host build of the device bodies of reprojection that follows moving geometry
// (crt_temporal_resampling_reprojected_motion, crt_restir_set_previous_triangles): tests/reuse/emu_reuse_reprojected.cpp
// (included unchanged) plus px_temporal with MOTION and the fused frame with px_candidate_temporal<..., REPROJ, RW, MOTION>,
// so that `pytest -m "not gpu"` checks them against the CPU specification (tests/reuse/reuse_port_motion.cpp).
#include "emu_reuse_reprojected.cpp"

namespace
{
template <class M, int RW>
void temporal_motion_all(int W, int H, int frame, const Bvh& bvh, const float* t, const crt_visibility* vis, f3 eye,
                         const Opt& o, const crt_raygen* prev_cam, const float* prev_t, const crt_visibility* prev_vis,
                         crt_reservoir* prev, crt_reservoir* res)
{
    launch(W, H, [&](Pix p)
           { px_temporal<M, RW, true>(p, frame, bvh, t, vis, eye, o, AosStore{prev}, AosStore{res}, prev_cam, W, H, prev_vis, prev_t); });
}
// k_candidate_temporal_reprojected<..., MOTION = true> + k_trace_shadow_queue<2>: the visibility-reuse rays traced inline
template <class M, int RW>
void candidate_temporal_motion_all(int W, int H, int frame, const Bvh& bvh, const float* t60, const crt_visibility* vis, f3 eye,
                                   const LightsIndexed& L, const Opt& opt, const SoaStore& T, const GBuf& g,
                                   const Reprojection& rp, const float* prev_t60)
{
    launch(W, H, [&](Pix p)
           {
               const DeferredRay d = px_candidate_temporal<M, LightsIndexed, true, RW, true>(
                   p, classify_pixel(p, t60, vis), frame, bvh, t60, eye, L, opt, T, g, HaloPeers(), 0u, rp, prev_t60);
               Hit h;
               if (d.want && !trace<true, true>(bvh, d.org, d.dir, 0.0f, 0.99f, h)) *T.mword(p.idx) |= kVisBit;
           });
}
}  // namespace

extern "C"
{
    // px_temporal with MOTION (crt_temporal_resampling_reprojected_motion)
    void rw_temporal_resampling_motion(int W, int H, int frame, void* gp, const crt_triangle* tris, int, const crt_visibility* vis,
                                       const float* eye, const crt_options* opt, const crt_raygen* prev_cam,
                                       const crt_triangle* prev_tris, const crt_visibility* prev_vis, const crt_reservoir* prev,
                                       crt_reservoir* res)
    {
        RW_CALL(temporal_motion_all, W, H, frame, ((EmuGeom*)gp)->view(), (const float*)tris, vis, v3(eye), make_opt(*opt),
                prev_cam, (const float*)prev_tris, prev_vis, (crt_reservoir*)prev, res);
    }

    // the fused frame with crt_restir_set_previous_frame (or, prev_vis null under the reference's weights,
    // crt_restir_set_previous_camera) and crt_restir_set_previous_triangles: rw_restir_frame_fast_reprojected's kernel
    // sequence with the motion candidate kernel; prev_tris == nullptr: rw_restir_frame_fast_reprojected itself
    void rw_restir_frame_fast_motion(int W, int H, int frame, void* gp, const crt_triangle* tris, const crt_raygen* rg,
                                     const float* eye_p, const uint32_t* lights, int nlights, const crt_options* options,
                                     crt_visibility* vis, char* temporal, char* res_a, char* res_b, crt_float4* accum,
                                     uint32_t* pixels, const crt_raygen* prev_rg, const crt_visibility* prev_vis,
                                     const crt_triangle* prev_tris)
    {
        if (!prev_rg || !prev_tris || !options->use_temporal_resampling)
        {
            rw_restir_frame_fast_reprojected(W, H, frame, gp, tris, rg, eye_p, lights, nlights, options, vis, temporal, res_a,
                                             res_b, accum, pixels, prev_rg, prev_vis);
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
        RW_CALL(candidate_temporal_motion_all, W, H, frame, bvh, t60, vis, eye, L, opt, T, g, rp, (const float*)prev_tris);
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
