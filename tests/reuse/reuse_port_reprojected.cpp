// TEST INFRASTRUCTURE — CPU specification of the unbiased reuse weights with a moving camera
// (crt_temporal_resampling_reprojected_surfaces, crt_restir_set_previous_frame; DESIGN.md section 15, "Reprojection").
// Built on the specification of the reuse weights (tests/reuse/reuse_port.cpp, included unchanged): the temporal merge
// with the history read at the port's reproject_pixel, its domain's surface taken from the previous frame's Visibility.
// The CUDA path (restir_core.cuh: temporal_merge_unbiased_reprojected, restir_pixel.cuh: px_temporal with a previous
// camera, restir_fast.cuh: px_candidate_temporal with REPROJ) restates it operation for operation.  Only tests/ load this.
#include "reuse_port.cpp"

namespace port
{
// The history is the previous frame's post-temporal reservoir at the reprojected pixel h and its domain's surface the
// previous frame's primary hit there — its Visibility record with the previous eye, the eye that frame's normals were
// flipped towards.  No history pixel, sky at h or M_h = 0: c_h = 0.
static void k_temporal_unbiased_reprojected(long tid, int W, int H, int frame, const Geom& g, const Visibility* vis, V3 eye,
                                            const Options& opt, const RayGen& prev_cam, const Visibility* prev_vis,
                                            const Reservoir* prev_buf, Reservoir* cur)
{
    const Px px = pixel_of(tid, W, H);
    const Visibility v = vis[px.idx];
    if (v.index == -1 || has_emission(g.tris[v.index])) return;
    if (!opt.use_temporal_resampling) return;
    Pcg rng(hash_pcg4(px.xi, px.yi, frame, 1), 0);
    const Surf surf = surface_from_visibility(v, g.tris, eye);
    int xp, yp;
    const bool found = reproject_pixel(prev_cam, W, H, surf.p, xp, yp);
    const int h = found ? xp + (H - yp - 1) * W : -1;
    Reservoir prev = found ? prev_buf[h] : empty_reservoir();
    Reservoir r = cur[px.idx];
    const int cap = 20 * opt.ris_sample_count;
    std::vector<Domain> domains{{surf, r.M}};
    int c_h = 0;
    if (found && prev.M > 0 && prev_vis[h].index != -1)
    {
        const Surf s_h = surface_from_visibility(prev_vis[h], g.tris, prev_cam.origin);
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
    // the reprojected temporal merge with the previous frame's Visibility; mode 0 is the port's reprojected k_temporal,
    // which does not read it
    void rw_temporal_resampling_reprojected(int W, int H, int frame, void* geom, const Triangle*, int, const Visibility* vis,
                                            const float* eye, const Options* opt, const RayGen* prev_cam,
                                            const Visibility* prev_vis, const Reservoir* prev, Reservoir* res)
    {
        const Geom& g = *(Geom*)geom;
        if (g_reuse_mode == kReuseUnbiased)
            launch(W, H, [&](long tid)
                   { k_temporal_unbiased_reprojected(tid, W, H, frame, g, vis, f3(eye), *opt, *prev_cam, prev_vis, prev, res); });
        else launch(W, H, [&](long tid) { k_temporal(tid, W, H, frame, g, vis, f3(eye), *opt, prev, res, prev_cam); });
    }
}
