// TEST INFRASTRUCTURE — CPU specification of power-proportional light selection (crt_set_light_sampling,
// CRT_LIGHTS_POWER; DESIGN.md section 14).  The reference has no counterpart, so this restatement is the specification and
// the CUDA path (csrc/restir_core.cuh: light_power .. slot_owner, geometry.cu: build_light_slots) restates it operation
// for operation.  It is built on the port of the reference (oracle/port/oracle_port.cpp, included unchanged): the light
// pick of generate_candidate, 08_nee and 09_ris goes through a LightSet, whose uniform mode is the reference's
// sample_light and 1.0f / size * 1.0f / area, and everything else is the port's own code.  Only tests/ load this library.
#include <vector>

#include "../../oracle/port/oracle_port.cpp"

namespace port
{
// ---- power-proportional light selection (extension, not in the reference; DESIGN.md section 14).  This is its
// specification: the CUDA table builder (csrc/restir_core.cuh: light_power .. slot_owner) restates it operation for
// operation.  Light i owns the slots [start_i, start_{i+1}) of a table of K = 2^k slots (n <= K <= 2^23): a candidate
// draws nth = (uint32)(rv0 * (float)K) exactly like the uniform pick draws over n, and light i is chosen with probability
// c_i / K, c_i = start_{i+1} - start_i >= 1.
//   P_i   = max(0, luminance(Le_i)) * area_i in float, non-finite -> 0
//   q_i   = (uint64) trunc((P_i / Pmax) * 2^32), all 0 when Pmax = 0
//   start_i = i + floor(R * S_i / S), S_i = sum_{j<i} q_j, S = S_n, R = K - n (128-bit product); S = 0: i + floor(R i / n)
// The record's selection probability is sel_i = (float)c_i * (1.0f / (float)K): with n = K every c_i = 1 and sel_i is
// 1.0f / (float)n, the uniform pdf, bit for bit.
constexpr int kLightsUniform = 0, kLightsPower = 1;
int g_light_mode = kLightsUniform;
int g_light_log2 = 0;  // 0: the default K
static float light_power(const Triangle& t)
{
    const float l = luminance(t.emissive);
    const float p = (l > 0.0f ? l : 0.0f) * area_of(t);
    return p <= kFltMax ? p : 0.0f;  // inf and NaN count as 0
}
// log2 K for n lights (-1: not a valid table size)
static int light_log2_slots(size_t n, int log2_slots)
{
    if (log2_slots == 0)
    {
        int c = 0;
        while (((size_t)1 << c) < n) c++;
        if (c > 23) return -1;  // more than 2^23 lights
        return c + 2 < 23 ? c + 2 : 23;
    }
    if (log2_slots < 0 || log2_slots > 23 || ((size_t)1 << log2_slots) < n) return -1;
    return log2_slots;
}
// start_0 .. start_n of the slot table; false when K is not valid for n
static bool light_starts(const Triangle* tris, const uint32_t* lights, size_t n, int log2_slots, std::vector<uint32_t>& start,
                         uint32_t& K)
{
    const int k = light_log2_slots(n, log2_slots);
    if (k < 0 || n == 0) return false;
    K = 1u << k;
    std::vector<float> P(n);
    float pmax = 0.0f;
    for (size_t i = 0; i < n; i++)
    {
        P[i] = light_power(tris[lights[i]]);
        pmax = P[i] > pmax ? P[i] : pmax;
    }
    const uint64_t R = K - (uint64_t)n;
    start.assign(n + 1, 0);
    uint64_t S = 0;
    std::vector<uint64_t> Si(n);
    for (size_t i = 0; i < n; i++)
    {
        Si[i] = S;
        S += pmax > 0.0f ? (uint64_t)((P[i] / pmax) * 4294967296.0f) : 0u;
    }
    for (size_t i = 0; i < n; i++)
        start[i] = (uint32_t)(i + (S ? (uint64_t)((unsigned __int128)R * Si[i] / S) : R * i / n));
    start[n] = K;
    return true;
}
// the lights as the samplers see them: the reference's list, plus the slot table in power mode
struct LightSet
{
    const uint32_t* lights;
    size_t n;
    bool power = false;
    uint32_t K = 0;
    std::vector<uint32_t> start;
};
static LightSet light_set(const Triangle* tris, const uint32_t* lights, size_t n)
{
    LightSet s;
    s.lights = lights;
    s.n = n;
    if (g_light_mode == kLightsPower && n) s.power = light_starts(tris, lights, n, g_light_log2, s.start, s.K);
    return s;
}
// the light that owns slot s: the last i with start_i <= s
static size_t slot_owner(const std::vector<uint32_t>& start, size_t n, uint32_t s)
{
    size_t lo = 0, hi = n - 1;
    while (lo < hi)
    {
        const size_t mid = (lo + hi + 1) / 2;
        if (start[mid] <= s) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}
static float slot_sel(const LightSet& s, size_t i) { return (float)(s.start[i + 1] - s.start[i]) * (1.0f / (float)s.K); }
// sample_light over a LightSet; `pdf` is what the reference divides by: 1.0f / size * 1.0f / area in uniform mode
static LightSample sample_light_set(const Triangle* tris, const LightSet& s, float rv0, float rv1, float rv2, float& pdf)
{
    if (!s.power)
    {
        const LightSample ls = sample_light(tris, s.lights, s.n, rv0, rv1, rv2);
        pdf = 1.0f / (float)s.n * 1.0f / area_of(tris[ls.index]);
        return ls;
    }
    uint32_t nth = (uint32_t)(rv0 * (float)s.K);
    if (nth == s.K) nth = s.K - 1;
    const size_t i = slot_owner(s.start, s.n, nth);
    LightSample ls;
    ls.index = (int)s.lights[i];
    const Triangle& t = tris[ls.index];
    ls.p = bary_point(t, warp_unit_triangle(rv1, rv2));
    ls.n = normal_of(t);
    pdf = slot_sel(s, i) * 1.0f / area_of(t);
    return ls;
}
// RIS over the emissive triangles (10_restir_di.cu:78-111, 09_ris.cu:66-100) with the light pick of a LightSet
static Reservoir ris_candidates_set(const Geom& g, const Surf& surf, const LightSet& lights, int count, bool shadowed, Pcg& rng)
{
    Reservoir r = empty_reservoir();
    for (int i = 0; i < count; ++i)
    {
        Sample s;
        memset(&s, 0, sizeof s);
        s.origin_position = surf.p;
        s.origin_normal = surf.n;
        float r0, r1, r2;
        draw3(rng, r0, r1, r2);
        float light_pdf;
        const LightSample ls = sample_light_set(g.tris, lights, r0, r1, r2, light_pdf);
        s.hit_position = ls.p;
        s.hit_normal = ls.n;
        const Triangle& lt = g.tris[ls.index];
        s.radiance = lt.emissive;
        const float p_hat = target_function(g, surf.p, surf.n, s.hit_position, s.hit_normal, s.radiance, shadowed);
        res_update(r, s, p_hat / light_pdf, rng.next_f());
    }
    return r;
}

// generate_candidate (10_restir_di.cu:36-135) with the light pick of a LightSet
static void k_generate_candidate_set(long tid, int W, int H, int frame, const Geom& g, const Visibility* vis, V3 eye,
                                 const LightSet& lights, const Options& opt,
                                 Reservoir* out)  // 10_restir_di.cu:36-135
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
    Reservoir r = ris_candidates_set(g, surf, lights, opt.ris_sample_count, false, rng);
    r.ucw = ucw_of(r, target_function(g, surf.p, surf.n, r.s.hit_position, r.s.hit_normal, r.s.radiance,
                                      opt.use_shadowed_target_function));
    if (opt.use_visibility_reuse) r.s.visibility = check_visibility(g, surf.p, surf.n, r.s.hit_position) != 0.0f;
    out[px.idx] = r;
}

// 08_nee / 09_ris (mode 8 / 9; 7 has no light pick) with the light pick of a LightSet
static void k_path_trace_set(long tid, int mode, int W, int H, int frame, const Geom& g, const LightSet& lights,
                         const RayGen& rg, const Options& opt, V4* accum)
{
    const Px px = pixel_of(tid, W, H);
    Pcg rng(hash_pcg3(px.xi, px.yi, frame), 0);
    V3 ro, rd;
    shoot(rg, (float)px.xi / (float)W, (float)px.yi / (float)H, ro, rd);
    V3 radiance = {0, 0, 0}, throughput = {1, 1, 1};
    for (int depth = 0; depth < opt.max_depth; ++depth)
    {
        Isect is;
        if (!raytrace(g, ro, rd, 0.0f, kFltMax, is))
        {
            if (mode == 7) radiance = radiance + throughput * opt.sky_color;
            break;
        }
        const Triangle& tri = g.tris[is.index];
        if (has_emission(tri))
        {
            if (mode == 7 || depth == 0) radiance = radiance + throughput * tri.emissive;
            break;
        }
        const Surf surf = surface_from_hit(ro, rd, is, g.tris);
        if (mode == 8)
        {
            float r0, r1, r2;
            draw3(rng, r0, r1, r2);
            float light_pdf;
            const LightSample ls = sample_light_set(g.tris, lights, r0, r1, r2, light_pdf);
            const Triangle& lt = g.tris[ls.index];
            const float V = check_visibility(g, surf.p, surf.n, ls.p);
            const V3 brdf = 1.0f / kPi * tri.color;
            const float G = geometry_term(surf.p, surf.n, ls.p, ls.n);
            radiance = radiance + throughput * brdf * G * V * lt.emissive / light_pdf;
        }
        else if (mode == 9)
        {
            const Reservoir r = ris_candidates_set(g, surf, lights, opt.ris_sample_count, opt.use_shadowed_target_function, rng);
            const V3 brdf = 1.0f / kPi * tri.color;
            const float G = geometry_term(surf.p, surf.n, r.s.hit_position, r.s.hit_normal);
            const float V = check_visibility(g, surf.p, surf.n, r.s.hit_position);
            const float p_hat = target_function(g, surf.p, surf.n, r.s.hit_position, r.s.hit_normal, r.s.radiance,
                                                opt.use_shadowed_target_function);
            radiance = radiance + throughput * brdf * G * V * r.s.radiance * ucw_of(r, p_hat);
        }
        const V3 wo = bounce_direction(surf, tri, rng);
        throughput = throughput * tri.color;
        ro = surf.p + 0.001f * surf.n;
        rd = wo;
    }
    accumulate(accum, px.idx, radiance, opt.accumulate);
}

}  // namespace port

extern "C"
{
    // light selection of ls_generate_candidate / ls_path_trace_mode: 0 uniform (the reference), 1 power-proportional
    // slots; log2_slots = 0: the default K.  A K that does not fit the light count makes ls_light_table return -1 (the
    // samplers then select uniformly, so callers check the table first).
    void ls_set_light_sampling(int mode, int log2_slots)
    {
        g_light_mode = mode;
        g_light_log2 = log2_slots;
    }
    // the K slot records of power mode (64 bytes each, the CUDA path's LightRec: v0, pdf, v1, n.x, v2, n.y, Le, n.z) into
    // `out` (capacity `cap` records; may be null to ask for K) and the n + 1 starts; returns K, or -1 when K does not fit n
    long ls_light_table(const Triangle* tris, const uint32_t* lights, int nlights, float* out, long cap, uint32_t* starts)
    {
        std::vector<uint32_t> start;
        uint32_t K = 0;
        if (!light_starts(tris, lights, (size_t)nlights, g_light_log2, start, K)) return -1;
        if (starts) memcpy(starts, start.data(), start.size() * sizeof(uint32_t));
        if (!out) return K;
        if (cap < (long)K) return -1;
        for (int i = 0; i < nlights; i++)
        {
            const Triangle& t = tris[lights[i]];
            const V3 c = cross(t.v[1] - t.v[0], t.v[2] - t.v[0]);
            const float len = length(c);
            const V3 nrm = c / len;
            const float sel = (float)(start[i + 1] - start[i]) * (1.0f / (float)K);
            const float rec[16] = {t.v[0].x, t.v[0].y, t.v[0].z, sel * 1.0f / (0.5f * len), t.v[1].x, t.v[1].y, t.v[1].z, nrm.x,
                                   t.v[2].x, t.v[2].y, t.v[2].z, nrm.y, t.emissive.x, t.emissive.y, t.emissive.z, nrm.z};
            for (uint32_t s = start[i]; s < start[i + 1]; s++) memcpy(out + 16 * (size_t)s, rec, sizeof rec);
        }
        return K;
    }
    // orc_generate_candidate with the light selection set above
    void ls_generate_candidate(int W, int H, int frame, void* geom, const Triangle*, int, const Visibility* vis,
                               const float* eye, const uint32_t* lights, int nlights, const Options* opt, Reservoir* res)
    {
        const Geom& g = *(Geom*)geom;
        const LightSet ls = light_set(g.tris, lights, nlights);
        launch(W, H, [&](long tid) { k_generate_candidate_set(tid, W, H, frame, g, vis, f3(eye), ls, *opt, res); });
    }
    // orc_path_trace_mode (8 or 9) with the light selection set above
    void ls_path_trace_mode(int mode, int W, int H, int frame, void* geom, const uint32_t* lights, int nlights,
                            const RayGen* rg, const Options* opt, V4* accum)
    {
        const Geom& g = *(Geom*)geom;
        const LightSet ls = light_set(g.tris, lights, nlights);
        launch(W, H, [&](long tid) { k_path_trace_set(tid, mode, W, H, frame, g, ls, *rg, *opt, accum); });
    }
}
