// TEST INFRASTRUCTURE — host build of the device bodies of the reuse weights (crt_set_reuse_weights): tests/emu's
// harness (included unchanged: the host BVH build, the orc_* kernels) plus the per-kernel and fused bodies with the reuse
// mode as their template parameter, so that `pytest -m "not gpu"` checks the CUDA path's arithmetic against the CPU
// specification (tests/reuse/reuse_port.cpp).
#include "../emu/emu.cpp"

namespace
{
int g_reuse_mode = CRT_REUSE_REFERENCE;
// fn<Math<0|1>, reuse mode>(args...) for the current math and reuse modes
#define RW_CALL(fn, ...)                                                                                                   \
    do {                                                                                                                   \
        const bool unb = g_reuse_mode == CRT_REUSE_UNBIASED;                                                               \
        if (g_math_mode) unb ? fn<Math<1>, CRT_REUSE_UNBIASED>(__VA_ARGS__) : fn<Math<1>, CRT_REUSE_REFERENCE>(__VA_ARGS__);  \
        else unb ? fn<Math<0>, CRT_REUSE_UNBIASED>(__VA_ARGS__) : fn<Math<0>, CRT_REUSE_REFERENCE>(__VA_ARGS__);              \
    } while (0)

template <class M, int RW>
void temporal_all(int W, int H, int frame, const Bvh& bvh, const float* t, const crt_visibility* vis, f3 eye, const Opt& o,
                  crt_reservoir* prev, crt_reservoir* res)
{
    launch(W, H, [&](Pix p) { px_temporal<M, RW>(p, frame, bvh, t, vis, eye, o, AosStore{prev}, AosStore{res}); });
}
template <class M, int RW>
void spatial_all(int W, int H, int frame, int pass, const Bvh& bvh, const float* t, const crt_visibility* vis, f3 eye,
                 const Opt& o, crt_reservoir* in, crt_reservoir* out)
{
    launch(W, H, [&](Pix p) { px_spatial<M, RW>(p, W, H, frame, pass, bvh, t, vis, eye, o, AosStore{in}, AosStore{out}); });
}
// k_candidate_temporal + k_trace_shadow_queue<2>: the visibility-reuse rays traced inline
template <class M, int RW>
void candidate_temporal_all(int W, int H, int frame, const Bvh& bvh, const float* t60, const crt_visibility* vis, f3 eye,
                            const LightsIndexed& L, const Opt& opt, const SoaStore& T, const GBuf& g)
{
    launch(W, H, [&](Pix p)
           {
               const DeferredRay d = px_candidate_temporal<M, LightsIndexed, false, RW>(p, classify_pixel(p, t60, vis), frame, bvh, t60,
                                                                                   eye, L, opt, T, g);
               Hit h;
               if (d.want && !trace<true, true>(bvh, d.org, d.dir, 0.0f, 0.99f, h)) *T.mword(p.idx) |= kVisBit;
           });
}
template <class M, int RW>
void spatial_fast_all(int W, int H, int frame, int pass, const Bvh& bvh, f3 eye, const Opt& opt, const SoaStore& in,
                      const SoaStore& out, const GBuf& g)
{
    launch(W, H, [&](Pix p) { px_spatial_fast<M, RW>(p, W, H, frame, pass, bvh, eye, opt, in, out, g); });
}
}  // namespace

extern "C"
{
    void rw_set_reuse_weights(int mode) { g_reuse_mode = mode; }
    // px_temporal / px_spatial (the per-kernel path: crt_temporal_resampling, crt_spatial_resampling)
    void rw_temporal_resampling(int W, int H, int frame, void* gp, const crt_triangle* tris, int, const crt_visibility* vis,
                                const float* eye, const crt_options* opt, const crt_reservoir* prev, crt_reservoir* res)
    {
        RW_CALL(temporal_all, W, H, frame, ((EmuGeom*)gp)->view(), (const float*)tris, vis, v3(eye), make_opt(*opt),
                (crt_reservoir*)prev, res);
    }
    void rw_spatial_resampling(int W, int H, int frame, int pass, void* gp, const crt_triangle* tris, int,
                               const crt_visibility* vis, const float* eye, const crt_options* opt, const crt_reservoir* in,
                               crt_reservoir* out)
    {
        RW_CALL(spatial_all, W, H, frame, pass, ((EmuGeom*)gp)->view(), (const float*)tris, vis, v3(eye), make_opt(*opt),
                (crt_reservoir*)in, out);
    }

    // the fused frame (csrc/kernels_fast.cu: crt_restir_di_frame) with the reuse mode: the kernel sequence of
    // emu_restir_frame_fast without reprojection
    void rw_restir_frame_fast(int W, int H, int frame, void* gp, const crt_triangle* tris, const crt_raygen* rg,
                              const float* eye_p, const uint32_t* lights, int nlights, const crt_options* options,
                              crt_visibility* vis, char* temporal, char* res_a, char* res_b, crt_float4* accum, uint32_t* pixels)
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
        const LightsIndexed L{t60, lights, (uint32_t)nlights};
        launch(W, H, [&](Pix p) { px_raycast(p, W, H, bvh, *rg, vis); });
        RW_CALL(candidate_temporal_all, W, H, frame, bvh, t60, vis, eye, L, opt, T, g);
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
