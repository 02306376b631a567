// TEST INFRASTRUCTURE — CPU specification of presampled light tiles (crt_set_light_tiles; DESIGN.md section 16).  The
// reference has no counterpart, so this restatement is the specification and the CUDA path (csrc/restir_core.cuh:
// light_tile_slot .. pixel_lights, geometry.cu: build_light_tiles) restates it operation for operation.  It is built on
// the light selection's specification (tests/lights/light_port.cpp, included unchanged): only generate_candidate's light
// pick changes, every other kernel is the port's own.  Only tests/ load this library.
//
//   source     the K records the candidates read without tiles: slot s is light s (uniform, K = n, sel = 1/n) or the
//              owner of slot s of the power table (K = 2^k, sel = c_i / K)
//   tile build entry e of tile t (T = 2^a tiles of S = 2^b entries) holds source slot
//                (uint32)(u * (float)K), u = next_f of Pcg(hash_pcg3(frame, t, e), 1), K - 1 if that is K
//   pixel      tile hash_pcg3(frame, xi >> 3, yi >> 2) & (T - 1)
//   candidate  nth = (uint32)(rv0 * (float)S), S - 1 if that is S; the light of tile[t][nth] with its source pdf
#include "light_port.cpp"

namespace port
{
int g_tiles_log2_t = 0, g_tiles_log2_s = 0;  // both 0: off

static uint32_t source_count(const LightSet& s) { return s.power ? s.K : (uint32_t)s.n; }
static uint32_t tile_slot(uint32_t frame, uint32_t t, uint32_t e, uint32_t K)
{
    Pcg rng(hash_pcg3(frame, t, e), 1);
    uint32_t s = (uint32_t)(rng.next_f() * (float)K);
    if (s == K) s = K - 1;
    return s;
}
static uint32_t tile_of(int xi, int yi, int frame, int log2_t)
{
    return hash_pcg3((uint32_t)frame, (uint32_t)xi >> 3, (uint32_t)yi >> 2) & ((1u << log2_t) - 1u);
}
// the light sample of source slot `slot` and the pdf its record carries
static LightSample sample_slot(const Triangle* tris, const LightSet& s, uint32_t slot, float rv1, float rv2, float& pdf)
{
    const size_t i = s.power ? slot_owner(s.start, s.n, slot) : slot;
    LightSample ls;
    ls.index = (int)s.lights[i];
    const Triangle& t = tris[ls.index];
    ls.p = bary_point(t, warp_unit_triangle(rv1, rv2));
    ls.n = normal_of(t);
    pdf = (s.power ? slot_sel(s, i) : 1.0f / (float)s.n) * 1.0f / area_of(t);
    return ls;
}
// generate_candidate (10_restir_di.cu:36-135) with the candidates drawn from the pixel's tile
static void k_generate_candidate_tiles(long tid, int W, int H, int frame, const Geom& g, const Visibility* vis, V3 eye,
                                       const LightSet& lights, const std::vector<uint32_t>& tiles, const Options& opt,
                                       Reservoir* out)
{
    const Px px = pixel_of(tid, W, H);
    const Visibility v = vis[px.idx];
    if (v.index == -1 || has_emission(g.tris[v.index]))
    {
        out[px.idx] = empty_reservoir();
        return;
    }
    Pcg rng(hash_pcg4(px.xi, px.yi, frame, 0), 0);
    const Surf surf = surface_from_visibility(v, g.tris, eye);
    const uint32_t S = 1u << g_tiles_log2_s;
    const uint32_t* tile = tiles.data() + (size_t)tile_of(px.xi, px.yi, frame, g_tiles_log2_t) * S;
    Reservoir r = empty_reservoir();
    for (int i = 0; i < opt.ris_sample_count; ++i)
    {
        Sample s;
        memset(&s, 0, sizeof s);
        s.origin_position = surf.p;
        s.origin_normal = surf.n;
        float r0, r1, r2;
        draw3(rng, r0, r1, r2);
        uint32_t nth = (uint32_t)(r0 * (float)S);
        if (nth == S) nth = S - 1;
        float light_pdf;
        const LightSample ls = sample_slot(g.tris, lights, tile[nth], r1, r2, light_pdf);
        s.hit_position = ls.p;
        s.hit_normal = ls.n;
        s.radiance = g.tris[ls.index].emissive;
        const float p_hat = target_function(g, surf.p, surf.n, s.hit_position, s.hit_normal, s.radiance, false);
        res_update(r, s, p_hat / light_pdf, rng.next_f());
    }
    r.ucw = ucw_of(r, target_function(g, surf.p, surf.n, r.s.hit_position, r.s.hit_normal, r.s.radiance,
                                      opt.use_shadowed_target_function));
    if (opt.use_visibility_reuse) r.s.visibility = check_visibility(g, surf.p, surf.n, r.s.hit_position) != 0.0f;
    out[px.idx] = r;
}
static std::vector<uint32_t> tile_slots(uint32_t K, int frame)
{
    const uint32_t S = 1u << g_tiles_log2_s, count = S << g_tiles_log2_t;
    std::vector<uint32_t> slots(count);
    for (uint32_t i = 0; i < count; i++) slots[i] = tile_slot((uint32_t)frame, i / S, i % S, K);
    return slots;
}
}  // namespace port

extern "C"
{
    void lt_set_light_tiles(int log2_tiles, int log2_tile_size)
    {
        g_tiles_log2_t = log2_tiles;
        g_tiles_log2_s = log2_tile_size;
    }
    // the source slots of the tiles of `frame` over K source records, T * S of them, tile t first at t * S
    void lt_tile_slots(uint32_t K, int frame, uint32_t* out)
    {
        const std::vector<uint32_t> s = tile_slots(K, frame);
        memcpy(out, s.data(), s.size() * sizeof(uint32_t));
    }
    // the tile of pixel (xi, yi) in `frame`
    uint32_t lt_tile_of(int xi, int yi, int frame) { return tile_of(xi, yi, frame, g_tiles_log2_t); }
    // ls_generate_candidate with light tiles (off: ls_generate_candidate itself)
    void lt_generate_candidate(int W, int H, int frame, void* geom, const Triangle* tris, int nt, const Visibility* vis,
                               const float* eye, const uint32_t* lights, int nlights, const Options* opt, Reservoir* res)
    {
        if ((!g_tiles_log2_t && !g_tiles_log2_s) || !nlights)
        {
            ls_generate_candidate(W, H, frame, geom, tris, nt, vis, eye, lights, nlights, opt, res);
            return;
        }
        const Geom& g = *(Geom*)geom;
        const LightSet ls = light_set(g.tris, lights, nlights);
        const std::vector<uint32_t> tiles = tile_slots(source_count(ls), frame);
        launch(W, H, [&](long tid) { k_generate_candidate_tiles(tid, W, H, frame, g, vis, f3(eye), ls, tiles, *opt, res); });
    }
}
