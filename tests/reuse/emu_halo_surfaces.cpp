// TEST INFRASTRUCTURE — host build of the halo-surface body of the fused frame on a row range (crt_restir_set_halo_surfaces,
// csrc/restir_fast.cuh: px_halo_surface) beside the candidate kernel's body (px_candidate_temporal, through
// tests/reuse/emu_reuse.cpp, included unchanged), so that `pytest -m "not gpu"` checks that a context which does not own a
// row writes the G-buffer record the row's owner writes, bit for bit.
#include "emu_reuse.cpp"

extern "C"
{
    // the G-buffer px_candidate_temporal writes for every pixel (g0: 16 B/px, g1: 8 B/px, cls: 1 B/px): the owners' records
    void hs_candidate_gbuf(int W, int H, int frame, void* gp, const crt_triangle* tris, const crt_visibility* vis,
                           const float* eye_p, const uint32_t* lights, int nlights, const crt_options* options, char* temporal,
                           char* g0, char* g1, uint8_t* cls)
    {
        const float* t60 = (const float*)tris;
        const LightsIndexed L{t60, lights, (uint32_t)nlights};
        const GBuf g{g0, g1, cls};
        RW_CALL(candidate_temporal_all, W, H, frame, ((EmuGeom*)gp)->view(), t60, vis, v3(eye_p), L, make_opt(*options),
                SoaStore{temporal, (size_t)W * H}, g);
    }
    // px_halo_surface over rows [y0, y1): what a context that does not own those rows writes
    void hs_halo_gbuf(int W, int H, int y0, int y1, const crt_triangle* tris, const crt_visibility* vis, const float* eye_p,
                      char* g0, char* g1, uint8_t* cls)
    {
        const GBuf g{g0, g1, cls};
        launch(W, H, [&](Pix p)
               {
                   if (p.yi >= y0 && p.yi < y1) px_halo_surface(p, (const float*)tris, vis, v3(eye_p), g);
               });
    }
}
