// TEST INFRASTRUCTURE — CPU specification of the unbiased reuse weights (crt_set_reuse_weights, CRT_REUSE_UNBIASED;
// DESIGN.md section 15).  The reference's reuse is biased by construction and has no unbiased mode, so this restatement is
// the specification and the CUDA path (csrc/restir_core.cuh: temporal_merge_unbiased .. ucw_unbiased, restir_pixel.cuh:
// px_temporal / px_spatial, restir_fast.cuh: px_candidate_temporal / spatial_fast_unbiased) restates it operation for
// operation.  It is built on the port of the reference (oracle/port/oracle_port.cpp, included unchanged through the light
// selection's specification tests/lights/light_port.cpp, so that candidates can also be drawn by power): k_temporal and
// k_spatial are restated with the weights below, and everything else is the port's own code.  Only tests/ load this library.
//
//   domain j       the pixel's own input reservoir and each accepted neighbour (spatial), or the pixel's current
//                  reservoir and its history (temporal); S_j is the primary-hit surface of domain j's *pixel*
//   c_j            trunc(M_j * rejection_heuristics(S_q, S_j)) — the reference's formula on two pixel surfaces; the
//                  temporal M cap applies first; the pixel's own domain has c = its input M
//   weight         p_hat_q(y_j) * ucw_j * c_j (the visibility bit multiplies nothing); selection and M as the reference's
//   Z              sum over domains of c_j [p_hat_j(y) > 0] for the selected sample y
//   ucw            p_hat_q(y) > 0 && Z > 0 ? w_sum / (Z * p_hat_q(y)) : 0
#include <vector>

#include "../lights/light_port.cpp"

namespace port
{
constexpr int kReuseReference = 0, kReuseUnbiased = 1;
int g_reuse_mode = kReuseReference;

// rejection_heuristics (reservoir.hpp:61-87) with the two pixel surfaces in place of the samples' origins
static float surface_heuristics(const Surf& s0, const Surf& s1, V3 eye)
{
    const float d0 = length(s0.p - eye);
    const float d1 = length(s1.p - eye);
    const float diff = (d1 - d0) * (d1 - d0) / d0;
    float w = 1.0f;
    w *= m_exp(-32.0f * diff);
    const float c = dot(s0.n, s1.n);
    w *= m_pow(c > 0.0f ? c : 0.0f, 8.0f);
    return w;
}
static int confidence(int m, const Surf& q, const Surf& j, V3 eye) { return to_int((float)m * surface_heuristics(q, j, eye)); }
static float p_hat_at(const Geom& g, const Surf& s, const Sample& y, bool shadowed)
{
    return target_function(g, s.p, s.n, y.hit_position, y.hit_normal, y.radiance, shadowed);
}
struct Domain
{
    Surf s;
    int c;
};
// Z and the unbiased contribution weight of the selected sample
static float ucw_unbiased(const Geom& g, const Surf& surf, const Reservoir& r, const std::vector<Domain>& domains, bool shadowed)
{
    const float p_hat = p_hat_at(g, surf, r.s, shadowed);
    long Z = 0;
    for (const Domain& d : domains)
        if (p_hat_at(g, d.s, r.s, shadowed) > 0.0f) Z += d.c;
    return p_hat > 0.0f && Z > 0 ? r.w_sum / ((float)Z * p_hat) : 0.0f;
}

static void k_temporal_unbiased(long tid, int W, int H, int frame, const Geom& g, const Visibility* vis, V3 eye,
                                const Options& opt, const Reservoir* prev_buf, Reservoir* cur)  // 10_restir_di.cu:137-237
{
    const Px px = pixel_of(tid, W, H);
    const Visibility v = vis[px.idx];
    if (v.index == -1 || has_emission(g.tris[v.index])) return;
    if (!opt.use_temporal_resampling) return;
    Pcg rng(hash_pcg4(px.xi, px.yi, frame, 1), 0);
    const Surf surf = surface_from_visibility(v, g.tris, eye);
    Reservoir prev = prev_buf[px.idx];
    Reservoir r = cur[px.idx];
    const int cap = 20 * opt.ris_sample_count;
    prev.M = prev.M < cap ? prev.M : cap;
    // the history's pixel is this pixel: without reprojection its surface is this frame's
    std::vector<Domain> domains{{surf, r.M}, {surf, confidence(prev.M, surf, surf, eye)}};
    const bool sh = opt.use_shadowed_target_function;
    prev.M = domains[1].c;
    res_merge(r, prev, p_hat_at(g, surf, prev.s, sh) * prev.ucw * (float)prev.M, rng.next_f());
    r.ucw = ucw_unbiased(g, surf, r, domains, sh);
    cur[px.idx] = r;
}

static void k_spatial_unbiased(long tid, int W, int H, int frame, int pass, const Geom& g, const Visibility* vis, V3 eye,
                               const Options& opt, const Reservoir* in, Reservoir* out)  // 10_restir_di.cu:256-388
{
    const Px px = pixel_of(tid, W, H);
    const Visibility v = vis[px.idx];
    if (v.index == -1 || has_emission(g.tris[v.index])) return;
    Pcg rng(hash_pcg4(px.xi, px.yi, frame, 2 + pass), 0);
    const Surf surf = surface_from_visibility(v, g.tris, eye);
    Reservoir r = in[px.idx];
    if (!opt.use_spatial_resampling)
    {
        out[px.idx] = r;
        return;
    }
    const bool sh = opt.use_shadowed_target_function;
    std::vector<Domain> domains{{surf, r.M}};
    for (int k = 0; k < opt.spatial_resampling_sample_count; ++k)
    {
        float rv0, rv1;
        draw2(rng, rv0, rv1);
        const V2 gs = sample_2d_gaussian(rv0, rv1);
        const int x = to_int((float)px.xi + opt.spatial_resampling_radius / 1.96f * gs.x);
        const int y = to_int((float)px.yi + opt.spatial_resampling_radius / 1.96f * gs.y);
        if (x < 0 || x >= W || y < 0 || y >= H) continue;
        if (x == px.xi && y == px.yi) continue;
        const int pid = x + (H - y - 1) * W;
        const Visibility nv = vis[pid];
        if (nv.index == -1 || has_emission(g.tris[nv.index])) continue;
        Reservoir nb = in[pid];
        const Surf ns = surface_from_visibility(nv, g.tris, eye);
        const Domain d{ns, confidence(nb.M, surf, ns, eye)};
        domains.push_back(d);
        nb.M = d.c;
        res_merge(r, nb, p_hat_at(g, surf, nb.s, sh) * nb.ucw * (float)nb.M, rng.next_f());
    }
    r.ucw = ucw_unbiased(g, surf, r, domains, sh);
    out[px.idx] = r;
}
}  // namespace port

extern "C"
{
    // 0: the reference's merges (the port's k_temporal / k_spatial), 1: unbiased weights
    void rw_set_reuse_weights(int mode) { g_reuse_mode = mode; }
    void rw_temporal_resampling(int W, int H, int frame, void* geom, const Triangle*, int, const Visibility* vis,
                                const float* eye, const Options* opt, const Reservoir* prev, Reservoir* res)
    {
        const Geom& g = *(Geom*)geom;
        if (g_reuse_mode == kReuseUnbiased)
            launch(W, H, [&](long tid) { k_temporal_unbiased(tid, W, H, frame, g, vis, f3(eye), *opt, prev, res); });
        else launch(W, H, [&](long tid) { k_temporal(tid, W, H, frame, g, vis, f3(eye), *opt, prev, res); });
    }
    void rw_spatial_resampling(int W, int H, int frame, int pass, void* geom, const Triangle*, int, const Visibility* vis,
                               const float* eye, const Options* opt, const Reservoir* in, Reservoir* out)
    {
        const Geom& g = *(Geom*)geom;
        if (g_reuse_mode == kReuseUnbiased)
            launch(W, H, [&](long tid) { k_spatial_unbiased(tid, W, H, frame, pass, g, vis, f3(eye), *opt, in, out); });
        else launch(W, H, [&](long tid) { k_spatial(tid, W, H, frame, pass, g, vis, f3(eye), *opt, in, out); });
    }
}
