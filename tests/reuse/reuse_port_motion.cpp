// TEST INFRASTRUCTURE — CPU specification of reprojection that follows moving geometry
// (crt_temporal_resampling_reprojected_motion, crt_restir_set_previous_triangles; DESIGN.md section 17).  Built on the
// specification of the reprojected reuse (tests/reuse/reuse_port_reprojected.cpp, included unchanged): the same merges,
// with the look-up at the point's previous position and, under unbiased weights, the history's surface on the triangle
// the previous frame saw.  The CUDA path (restir_pixel.cuh: previous_point, previous_surface<true>, px_temporal with
// MOTION; restir_fast.cuh: px_candidate_temporal with MOTION) restates it operation for operation.  Only tests/ load this.
#include <cstring>

#include "reuse_port_reprojected.cpp"

namespace port
{
// the 36 vertex bytes of triangle i differ between the two arrays
static bool moved(const Triangle* tris, const Triangle* prev_tris, int i)
{
    return memcmp(tris[i].v, prev_tris[i].v, sizeof tris[i].v) != 0;
}
// 1. the point's previous position: the surface point itself on an unmoved triangle, otherwise the same barycentrics on
// the previous vertices; then the look-up as today.  h = -1: no history.
static int history_pixel(int W, int H, const Visibility& v, const Surf& surf, const Triangle* tris, const Triangle* prev_tris,
                         const RayGen& prev_cam)
{
    const V3 p_prev = moved(tris, prev_tris, v.index) ? bary_point(prev_tris[v.index], v.uv) : surf.p;
    int xp, yp;
    return reproject_pixel(prev_cam, W, H, p_prev, xp, yp) ? xp + (H - yp - 1) * W : -1;
}

// reference weights: the port's k_temporal with a previous camera, the history read at history_pixel
static void k_temporal_motion(long tid, int W, int H, int frame, const Geom& g, const Visibility* vis, V3 eye,
                              const Options& opt, const Reservoir* prev_buf, Reservoir* cur, const RayGen& prev_cam,
                              const Triangle* prev_tris)
{
    const Px px = pixel_of(tid, W, H);
    const Visibility v = vis[px.idx];
    if (v.index == -1 || has_emission(g.tris[v.index])) return;
    if (!opt.use_temporal_resampling) return;
    Pcg rng(hash_pcg4(px.xi, px.yi, frame, 1), 0);
    const Surf surf = surface_from_visibility(v, g.tris, eye);
    const int h = history_pixel(W, H, v, surf, g.tris, prev_tris, prev_cam);
    Reservoir prev = h >= 0 ? prev_buf[h] : empty_reservoir();
    Reservoir r = cur[px.idx];
    const int cap = 20 * opt.ris_sample_count;
    prev.M = prev.M < cap ? prev.M : cap;
    float p_hat_y = target_function(g, surf.p, surf.n, prev.s.hit_position, prev.s.hit_normal, prev.s.radiance,
                                    opt.use_shadowed_target_function);
    if (opt.use_visibility_reuse) p_hat_y *= (float)prev.s.visibility;
    prev.M = to_int((float)prev.M * rejection_heuristics(r, prev, eye));
    const float weight = p_hat_y * prev.ucw * (float)prev.M;
    res_merge(r, prev, weight, rng.next_f());
    r.ucw = ucw_of(r, target_function(g, surf.p, surf.n, r.s.hit_position, r.s.hit_normal, r.s.radiance,
                                      opt.use_shadowed_target_function));
    cur[px.idx] = r;
}

// unbiased weights: k_temporal_unbiased_reprojected with the history read at history_pixel and S_h built on the
// previous array's triangle when that triangle moved, on this frame's otherwise (2.)
static void k_temporal_unbiased_motion(long tid, int W, int H, int frame, const Geom& g, const Visibility* vis, V3 eye,
                                       const Options& opt, const RayGen& prev_cam, const Triangle* prev_tris,
                                       const Visibility* prev_vis, const Reservoir* prev_buf, Reservoir* cur)
{
    const Px px = pixel_of(tid, W, H);
    const Visibility v = vis[px.idx];
    if (v.index == -1 || has_emission(g.tris[v.index])) return;
    if (!opt.use_temporal_resampling) return;
    Pcg rng(hash_pcg4(px.xi, px.yi, frame, 1), 0);
    const Surf surf = surface_from_visibility(v, g.tris, eye);
    const int h = history_pixel(W, H, v, surf, g.tris, prev_tris, prev_cam);
    Reservoir prev = h >= 0 ? prev_buf[h] : empty_reservoir();
    Reservoir r = cur[px.idx];
    const int cap = 20 * opt.ris_sample_count;
    std::vector<Domain> domains{{surf, r.M}};
    int c_h = 0;
    if (h >= 0 && prev.M > 0 && prev_vis[h].index != -1)
    {
        const Triangle* t = moved(g.tris, prev_tris, prev_vis[h].index) ? prev_tris : g.tris;
        const Surf s_h = surface_from_visibility(prev_vis[h], t, prev_cam.origin);
        c_h = confidence(prev.M < cap ? prev.M : cap, surf, s_h, eye);
        domains.push_back({s_h, c_h});
    }
    const bool shadowed = opt.use_shadowed_target_function;
    prev.M = c_h;
    res_merge(r, prev, p_hat_at(g, surf, prev.s, shadowed) * prev.ucw * (float)prev.M, rng.next_f());
    r.ucw = ucw_unbiased(g, surf, r, domains, shadowed);
    cur[px.idx] = r;
}
}  // namespace port

extern "C"
{
    // the reprojected temporal merge that follows moving geometry; prev_tris: the previous frame's triangle array (the
    // same count and order as the geometry's); prev_vis is read under unbiased weights only
    void rw_temporal_resampling_motion(int W, int H, int frame, void* geom, const Triangle*, int, const Visibility* vis,
                                       const float* eye, const Options* opt, const RayGen* prev_cam, const Triangle* prev_tris,
                                       const Visibility* prev_vis, const Reservoir* prev, Reservoir* res)
    {
        const Geom& g = *(Geom*)geom;
        if (g_reuse_mode == kReuseUnbiased)
            launch(W, H, [&](long tid)
                   { k_temporal_unbiased_motion(tid, W, H, frame, g, vis, f3(eye), *opt, *prev_cam, prev_tris, prev_vis, prev, res); });
        else launch(W, H, [&](long tid) { k_temporal_motion(tid, W, H, frame, g, vis, f3(eye), *opt, prev, res, *prev_cam, prev_tris); });
    }
}
