// restir_core.cuh — per-pixel logic of the ReSTIR DI path (examples 06-10), layout-agnostic.
// The kernels (kernels_*.cu) decide how reservoirs are stored (reference AoS or SoA planes) and hand
// register-resident values to these functions.  Every function cites the reference lines it implements;
// arithmetic order follows the reference exactly (see vecmath.cuh for the numerics contract).
#pragma once
#include "bvh.cuh"

namespace crt
{
#if defined(__CUDA_ARCH__)
#define CRT_LDG(p) __ldg(p)
#else
#define CRT_LDG(p) (*(p))
#endif

// ---- reference Triangle (common/core.hpp:38-43): 15 floats, 60-byte stride, 4-byte aligned
struct TriRef
{
    const float* p;
    CRT_HD f3 v(int k) const { return {CRT_LDG(p + 3 * k), CRT_LDG(p + 3 * k + 1), CRT_LDG(p + 3 * k + 2)}; }
    CRT_HD f3 color() const { return {CRT_LDG(p + 9), CRT_LDG(p + 10), CRT_LDG(p + 11)}; }
    CRT_HD f3 emissive() const { return {CRT_LDG(p + 12), CRT_LDG(p + 13), CRT_LDG(p + 14)}; }
};
CRT_HD TriRef tri_at(const float* tris60, int index) { return TriRef{tris60 + (size_t)index * 15}; }
CRT_HD bool has_emission(f3 e) { return e.x > 0.0f || e.y > 0.0f || e.z > 0.0f; }  // core.hpp:65-69
CRT_HD f3 tri_normal(f3 v0, f3 v1, f3 v2) { return normalize(cross(v1 - v0, v2 - v0)); }      // core.hpp:50-55
CRT_HD float tri_area(f3 v0, f3 v1, f3 v2) { return 0.5f * length(cross(v1 - v0, v2 - v0)); }  // core.hpp:57-62
CRT_HD f3 bary_point(f3 v0, f3 v1, f3 v2, float u, float v) { return (1.0f - u - v) * v0 + u * v1 + v * v2; }

// ---- camera (common/camera.hpp:27-35); pixel -> (u,v) = (xi/W, yi/H) as in 10_restir_di.cu:24
struct RayGen
{
    f3 origin, right, up;
};
CRT_HD void shoot(const RayGen& rg, float u, float v, f3& ro, f3& rd)
{
    const f3 forward = normalize(cross(rg.up, rg.right));
    const f3 to = rg.origin + forward + mix(-rg.right, rg.right, u) + mix(rg.up, -rg.up, v);
    ro = rg.origin;
    rd = normalize(to - rg.origin);
}

// ---- temporal reprojection (extension, SURVEY.md section 8 f2; the specification is the checker's reproject_pixel — see
// DESIGN.md section 11 — restated here operation for operation).  The inverse of shoot(): to = o + forward + right (2u - 1) + up (1 - 2v); the
// pixel whose sample point (xi / W, yi / H) is nearest to the projection of `p` in the previous frame's camera.
CRT_HD bool reproject_pixel(const RayGen& prev, int W, int H, f3 p, int& xp, int& yp)
{
    const f3 forward = normalize(cross(prev.up, prev.right));
    const f3 d = p - prev.origin;
    const float s = dot(d, forward);
    if (!(s > 0.0f)) return false;
    const f3 q = d / s;
    const float a = dot(q, prev.right) / dot(prev.right, prev.right);
    const float b = dot(q, prev.up) / dot(prev.up, prev.up);
    const float u = (a + 1.0f) * 0.5f;
    const float v = (1.0f - b) * 0.5f;
    xp = f2i_trunc(floorf(u * (float)W + 0.5f));
    yp = f2i_trunc(floorf(v * (float)H + 0.5f));
    return xp >= 0 && xp < W && yp >= 0 && yp < H;
}

// ---- raytrace.hpp:45-52 — origin p0 + 1e-3 n0 (core.hpp:32-36), direction p1 - p0 (not renormalised),
// t in [0, 0.99]; the reference asks for the closest hit but only uses hit / no hit -> any-hit walk.
CRT_HD float check_visibility(const Bvh& bvh, f3 p0, f3 n0, f3 p1)
{
    Hit h;
    return trace<true, true>(bvh, p0 + 0.001f * n0, p1 - p0, 0.0f, 0.99f, h) ? 0.0f : 1.0f;  // towards a light: far end first
}

// ---- surfaces (core.hpp:188-207 and 152-165)
struct Surf
{
    f3 p, n;
};
CRT_HD Surf surface_from_visibility(const TriRef& t, float u, float v, f3 eye)
{
    const f3 v0 = t.v(0), v1 = t.v(1), v2 = t.v(2);
    Surf s{bary_point(v0, v1, v2, u, v), tri_normal(v0, v1, v2)};
    const f3 view = normalize(eye - s.p);
    if (dot(view, s.n) < 0.0f) s.n = -s.n;
    return s;
}
CRT_HD Surf surface_from_hit(const TriRef& t, f3 ro, f3 rd, float thit)
{
    Surf s{ro + thit * rd, tri_normal(t.v(0), t.v(1), t.v(2))};
    if (dot(-rd, s.n) < 0.0f) s.n = -s.n;
    return s;
}

// ---- sampling (core.hpp:76-89, 237-295)
template <class M>
CRT_HD f3 sample_hemisphere(float r0, float r1, float r2)
{
    const float theta = r0 * 2.0f * kPi;
    float radius = r1 + r2;
    if (1.0f < radius) radius = 2.0f - radius;
    const float x = M::cos(theta) * radius;
    const float z = M::sin(theta) * radius;
    const float yy = 1.0f - radius * radius;
    return {x, sqrtf(yy < 0.0f ? 0.0f : yy), z};
}
CRT_HD f2 warp_unit_triangle(float x, float y)  // Heitz 2019, core.hpp:237-252
{
    if (y > x) { x *= 0.5f; y -= x; }
    else { y *= 0.5f; x -= y; }
    return {x, y};
}
struct LightSample
{
    f3 p, n, emissive;
    float area;
    float pdf;  // LightsTable only: 1.0f / size * 1.0f / area (10_restir_di.cu:98-99), divided once when the table is built
};
// core.hpp:261-285 plus what the callers read from the same triangle (emissive, area_of).
// Two interchangeable sources with identical results:
//   LightsIndexed  the reference's double indirection lights[nth] -> triangles[index] (60-byte AoS gather)
//   LightsTable    a 64-byte record per light, built once per (geometry, light list): vertices, the normal and
//                  area the reference recomputes per candidate (same operations, so the same bits), emission
struct LightsIndexed
{
    const float* tris60;
    const uint32_t* lights;
    uint32_t n;
    static constexpr bool kHasPdf = false;
    struct Raw
    {
        const float* tri;
    };
    CRT_HD Raw fetch(float rv0, unsigned /*pair_mask*/ = 0u) const
    {
        uint32_t nth = (uint32_t)(rv0 * (float)n);
        if (nth == n) nth = n - 1;
        return Raw{tris60 + (size_t)CRT_LDG(lights + nth) * 15};
    }
    CRT_HD LightSample finish(const Raw& raw, float rv1, float rv2) const
    {
        const TriRef t{raw.tri};
        const f3 v0 = t.v(0), v1 = t.v(1), v2 = t.v(2);
        const f2 b = warp_unit_triangle(rv1, rv2);
        LightSample ls;
        ls.p = bary_point(v0, v1, v2, b.x, b.y);
        const f3 c = cross(v1 - v0, v2 - v0);
        const float len = length(c);
        ls.n = c / len;        // normal_of
        ls.area = 0.5f * len;  // area_of
        ls.pdf = 0.0f;
        ls.emissive = t.emissive();
        return ls;
    }
    CRT_HD LightSample sample(float rv0, float rv1, float rv2) const { return finish(fetch(rv0), rv1, rv2); }
    using Elem = uint32_t;
    static CRT_HD LightsIndexed at(const float* tris60, const uint32_t* lights, uint32_t n) { return LightsIndexed{tris60, lights, n}; }
};
struct alignas(16) LightRec  // 64 bytes
{
    float v0x, v0y, v0z, pdf;  // pdf = 1.0f / size * 1.0f / area: what every candidate divides by (saves one of its seven IEEE divisions)
    float v1x, v1y, v1z, nx;
    float v2x, v2y, v2z, ny;
    float ex, ey, ez, nz;
};
// the record of a light selected with probability `sel`
CRT_HD LightRec light_rec(const float* tris60, uint32_t tri_index, float sel)
{
    const TriRef t = tri_at(tris60, (int)tri_index);
    const f3 v0 = t.v(0), v1 = t.v(1), v2 = t.v(2), e = t.emissive();
    const f3 c = cross(v1 - v0, v2 - v0);
    const float len = length(c);
    const f3 n = c / len;
    return LightRec{v0.x, v0.y, v0.z, sel * 1.0f / (0.5f * len), v1.x, v1.y, v1.z, n.x, v2.x, v2.y, v2.z, n.y, e.x, e.y, e.z, n.z};
}
// the uniform record, sel = 1/n (kept as its own function: written through light_rec, nvcc schedules the division
// differently and k_build_light_table's SASS changes)
CRT_HD LightRec make_light_rec(const float* tris60, uint32_t tri_index, uint32_t n_lights)
{
    const TriRef t = tri_at(tris60, (int)tri_index);
    const f3 v0 = t.v(0), v1 = t.v(1), v2 = t.v(2), e = t.emissive();
    const f3 c = cross(v1 - v0, v2 - v0);
    const float len = length(c);
    const f3 n = c / len;
    const float inv_n = 1.0f / (float)n_lights;  // as ris_candidates computes it
    return LightRec{v0.x, v0.y, v0.z, inv_n * 1.0f / (0.5f * len), v1.x, v1.y, v1.z, n.x, v2.x, v2.y, v2.z, n.y, e.x, e.y, e.z, n.z};
}

// ---- power-proportional light selection (crt_set_light_sampling, CRT_LIGHTS_POWER; DESIGN.md section 14).  Light i
// owns the slots [start_i, start_{i+1}) of a table of K = 2^k slots, n <= K <= 2^23, and slot s holds light_rec(...,
// slot_sel(c_i, K)), c_i = start_{i+1} - start_i >= 1.  LightsTable{slots, K} draws nth = (uint32)(rv0 * (float)K): rv0
// is a multiple of 2^-23, so every slot has probability exactly 1/K and light i exactly c_i / K, the record's `sel`.
// The slot counts are computed in integers from quantised powers, so that they do not depend on summation order: the
// host's restatement (the CPU specification) and this device build produce the same table bit for bit.
constexpr int kMaxLightSlotsLog2 = 23;
// log2 K for n lights: requested (1..23, 2^k >= n) or, for 0, min(23, ceil(log2 n) + 2); -1 when none fits
CRT_HD int light_slots_log2(uint64_t n, int requested)
{
    if (requested == 0)
    {
        int c = 0;
        while (((uint64_t)1 << c) < n) c++;
        if (c > kMaxLightSlotsLog2) return -1;  // more than 2^23 lights
        return c + 2 < kMaxLightSlotsLog2 ? c + 2 : kMaxLightSlotsLog2;
    }
    if (requested < 0 || requested > kMaxLightSlotsLog2 || ((uint64_t)1 << requested) < n) return -1;
    return requested;
}
// P_i = max(0, luminance(Le_i)) * area_i; non-finite -> 0 (so every value compares as an unsigned integer)
CRT_HD float light_power(const float* tris60, uint32_t tri_index)
{
    const TriRef t = tri_at(tris60, (int)tri_index);
    const float l = luminance(t.emissive());
    const float p = (l > 0.0f ? l : 0.0f) * tri_area(t.v(0), t.v(1), t.v(2));
    return p <= kFltMax ? p : 0.0f;
}
// q_i = trunc((P_i / Pmax) * 2^32)
CRT_HD uint64_t light_quantum(float p, float pmax) { return pmax > 0.0f ? (uint64_t)((p / pmax) * 4294967296.0f) : 0u; }
// start_i = i + floor(R * S_i / S), R = K - n, S_i = sum_{j<i} q_j (R S_i < 2^78: 128-bit); S = 0: i + floor(R i / n)
CRT_HD uint32_t light_start(uint32_t i, uint32_t n, uint32_t K, uint64_t s_i, uint64_t s)
{
    const uint64_t R = (uint64_t)K - n;
    return i + (uint32_t)(s ? (uint64_t)((unsigned __int128)R * s_i / s) : R * i / n);
}
// the light that owns slot s: the last i with start[i] <= s (start[0] = 0, strictly increasing)
CRT_HD uint32_t slot_owner(const uint32_t* start, uint32_t n, uint32_t s)
{
    uint32_t lo = 0, hi = n - 1;
    while (lo < hi)
    {
        const uint32_t mid = lo + (hi - lo + 1) / 2;
        if (CRT_LDG(start + mid) <= s) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}
CRT_HD float slot_sel(uint32_t c, uint32_t K) { return (float)c * (1.0f / (float)K); }
struct LightsTable
{
    const LightRec* table;
    uint32_t n;
    static constexpr bool kHasPdf = true;
    struct Raw
    {
        u4 a, b, c, d;
    };
    // the gather, separated from the arithmetic so that callers can have several records in flight.
    //
    // pair_mask != 0 (device only): the lanes named in it call fetch together, and with it each lane 2k and its
    // neighbour 2k+1 are both named.  The two then share their gathers: the L1 charges one wavefront per distinct
    // 128-byte line per load instruction, a 64-byte record needs two 256-bit loads, so a warp fetching 32 records on
    // its own pays 64 wavefronts.  Paired, both lanes read the even lane's record in the first instruction (one
    // half each) and the odd lane's in the second: 32 wavefronts, and the halves that landed in the partner's
    // registers come back through eight shuffles.
    // MEASURED AND REJECTED (profiles/r1/bench_o_pair_gather.json): k_candidate_temporal 2.19 -> 3.08 ms at 4K.  The
    // loop issues 63 % of its cycles and the nine extra SHFL per candidate (2.26 G warp instructions against
    // 1.76 G) cost more than the halved tag traffic saves.  Kept behind CRT_LIGHT_PAIR for the record.
    CRT_HD Raw fetch(float rv0, unsigned pair_mask = 0u) const
    {
        uint32_t nth = (uint32_t)(rv0 * (float)n);
        if (nth == n) nth = n - 1;
#if defined(__CUDA_ARCH__) && defined(CRT_LIGHT_PAIR) && !defined(CRT_LIGHT_LDG128)
        const unsigned lane = threadIdx.x & 31u;
        if ((pair_mask >> lane) & 1u)
        {
            const bool odd = (lane & 1u) != 0u;
            const uint32_t other = __shfl_xor_sync(pair_mask, nth, 1);
            const char* half = (const char*)table + (odd ? 32 : 0);
            const u8w x = load_u8w(half + (size_t)(odd ? other : nth) * 64);  // the even lane's record
            const u8w y = load_u8w(half + (size_t)(odd ? nth : other) * 64);  // the odd lane's record
            // even keeps x (low half of its record) and is owed the high half = odd's x; odd keeps y (high half) and
            // is owed the low half = even's y
            const u8w send = odd ? x : y;
            u8w recv;
            recv.lo.x = __shfl_xor_sync(pair_mask, send.lo.x, 1);
            recv.lo.y = __shfl_xor_sync(pair_mask, send.lo.y, 1);
            recv.lo.z = __shfl_xor_sync(pair_mask, send.lo.z, 1);
            recv.lo.w = __shfl_xor_sync(pair_mask, send.lo.w, 1);
            recv.hi.x = __shfl_xor_sync(pair_mask, send.hi.x, 1);
            recv.hi.y = __shfl_xor_sync(pair_mask, send.hi.y, 1);
            recv.hi.z = __shfl_xor_sync(pair_mask, send.hi.z, 1);
            recv.hi.w = __shfl_xor_sync(pair_mask, send.hi.w, 1);
            const u8w lo = odd ? recv : x, hi = odd ? y : recv;
            return Raw{lo.lo, lo.hi, hi.lo, hi.hi};
        }
#endif
        const char* q = (const char*)(table + nth);
#if defined(CRT_LIGHT_LDG128)
        return Raw{load_u4(q), load_u4(q + 16), load_u4(q + 32), load_u4(q + 48)};
#else
        const u8w lo = load_u8w(q), hi = load_u8w(q + 32);  // two 256-bit requests per record
        return Raw{lo.lo, lo.hi, hi.lo, hi.hi};
#endif
    }
    CRT_HD LightSample finish(const Raw& raw, float rv1, float rv2) const
    {
        const u4 &a = raw.a, &b4 = raw.b, &c4 = raw.c, &d = raw.d;
        const f3 v0{u2f(a.x), u2f(a.y), u2f(a.z)}, v1{u2f(b4.x), u2f(b4.y), u2f(b4.z)}, v2{u2f(c4.x), u2f(c4.y), u2f(c4.z)};
        const f2 b = warp_unit_triangle(rv1, rv2);
        LightSample ls;
        ls.p = bary_point(v0, v1, v2, b.x, b.y);
        ls.n = f3{u2f(b4.w), u2f(c4.w), u2f(d.w)};
        ls.area = 0.0f;  // folded into pdf
        ls.pdf = u2f(a.w);
        ls.emissive = f3{u2f(d.x), u2f(d.y), u2f(d.z)};
        return ls;
    }
    CRT_HD LightSample sample(float rv0, float rv1, float rv2) const { return finish(fetch(rv0), rv1, rv2); }
    using Elem = LightRec;
    static CRT_HD LightsTable at(const float*, const LightRec* table, uint32_t n) { return LightsTable{table, n}; }
};
// the pdf the reference divides a light sample by: 1.0f / size * 1.0f / area (08_nee.cu, 10_restir_di.cu:98-99), or the
// record's own (LightsTable)
template <class L>
CRT_HD float light_pdf_of(const LightSample& ls, uint32_t n)
{
    return L::kHasPdf ? ls.pdf : 1.0f / (float)n * 1.0f / ls.area;
}

// ---- presampled light tiles (crt_set_light_tiles; DESIGN.md section 16).  Once per frame T = 2^log2_t tiles of
// S = 2^log2_s records are drawn from the source table (K records: one per light, or the slot table of CRT_LIGHTS_POWER):
// entry e of tile t copies record light_tile_slot(frame, t, e, K), pdf included.  A pixel's candidates draw from the one
// tile of its 8x4 block (light_tile_of: one warp of tile_grid reads one tile), nth = (uint32)(rv0 * (float)S): entries
// are uniform, and every entry is marginally distributed like a candidate drawn from the source, so each candidate is too.
// the source slot of entry e of tile t: drawn from a stream of its own as a candidate draws rv0 (LightsTable::fetch)
CRT_HD uint32_t light_tile_slot(uint32_t frame, uint32_t t, uint32_t e, uint32_t K)
{
    Pcg rng(hash_pcg3(frame, t, e), 1);
    uint32_t s = (uint32_t)(rng.next_f() * (float)K);
    if (s == K) s = K - 1;
    return s;
}
// the tile of pixel (xi, yi), in global pixel coordinates (every row range agrees); reads no pixel's random stream
CRT_HD uint32_t light_tile_of(int xi, int yi, int frame, uint32_t log2_t)
{
    return hash_pcg3((uint32_t)frame, (uint32_t)xi >> 3, (uint32_t)yi >> 2) & ((1u << log2_t) - 1u);
}
struct LightsTiles
{
    const LightRec* tiles;  // T * S records, tile t at tiles + t * S
    uint32_t log2_t, log2_s;
};
// the light source a pixel's candidates draw from: the source itself, or with tiles a LightsTable over the pixel's tile
template <class L>
CRT_HD const L& pixel_lights(const L& lights, int, int, int) { return lights; }
CRT_HD LightsTable pixel_lights(const LightsTiles& lights, int xi, int yi, int frame)
{
    return LightsTable{lights.tiles + ((size_t)light_tile_of(xi, yi, frame, lights.log2_t) << lights.log2_s), 1u << lights.log2_s};
}
CRT_HD float geometry_term(f3 p0, f3 n0, f3 p1, f3 n1)  // core.hpp:287-295
{
    f3 v = p1 - p0;
    const float sqr = dot(v, v);
    v = normalize(v);
    return fabsf(dot(v, n0)) * fabsf(dot(-v, n1)) / sqr;
}

// ---- reservoir (common/reservoir.hpp)
struct Sample
{
    f3 op, on, hp, hn, rad;  // origin position/normal, hit position/normal, radiance
    uint32_t vis;            // bit 0: bool visibility; bit 1 (fused frame only): traced, see restir_fast.cuh kSampleTraced
};
struct Res
{
    Sample s;
    float w_sum, ucw;
    int M;
};
CRT_HD Res empty_res()
{
    Res r;
    r.s.op = r.s.on = r.s.hp = r.s.hn = r.s.rad = f3{0.0f, 0.0f, 0.0f};
    r.s.vis = 0;
    r.w_sum = r.ucw = 0.0f;
    r.M = 0;
    return r;
}
CRT_HD float target_function(const Bvh& bvh, f3 p0, f3 n0, f3 p1, f3 n1, f3 radiance, bool shadowed)  // :42-59
{
    const float G = geometry_term(p0, n0, p1, n1);
    if (shadowed) return kInvPi * G * check_visibility(bvh, p0, n0, p1) * luminance(radiance);
    return kInvPi * G * luminance(radiance);
}
template <class M>
CRT_HD float rejection_heuristics(const Sample& s0, const Sample& s1, f3 eye)  // reservoir.hpp:61-87
{
    const float d0 = length(s0.op - eye);
    const float d1 = length(s1.op - eye);
    const float diff = (d1 - d0) * (d1 - d0) / d0;
    float w = 1.0f;
    w *= M::exp(-32.0f * diff);
    const float c = dot(s0.on, s1.on);
    w *= M::pow(c > 0.0f ? c : 0.0f, 8.0f);
    return w;
}
template <class M>
CRT_HD f2 sample_2d_gaussian(float rv0, float rv1)  // reservoir.hpp:89-95
{
    const float a = -2.0f * M::log(rv0);
    const float radius = sqrtf(a > 0.0f ? a : 0.0f);
    const float phi = 2.0f * kPi * rv1;
#if defined(__CUDA_ARCH__) && !defined(CRT_NO_SINCOS)
    float s, c;
    M::sincos(phi, s, c);
    return {radius * c, radius * s};
#else
    return {radius * M::cos(phi), radius * M::sin(phi)};
#endif
}
CRT_HD float ucw_of(const Res& r, float p_hat) { return p_hat > 0.0f ? r.w_sum / ((float)r.M * p_hat) : 0.0f; }

struct Opt  // the fields of common/options.hpp:4-23 the kernels read
{
    bool accumulate, temporal, spatial, shadowed, reuse;
    int max_depth, ris_count, spatial_count;
    float radius;
    f3 sky;
};
CRT_HD Opt make_opt(const crt_options& o)
{
    Opt r;
    r.accumulate = o.accumulate != 0;
    r.temporal = o.use_temporal_resampling != 0;
    r.spatial = o.use_spatial_resampling != 0;
    r.shadowed = o.use_shadowed_target_function != 0;
    r.reuse = o.use_visibility_reuse != 0;
    r.max_depth = o.max_depth;
    r.ris_count = o.ris_sample_count;
    r.spatial_count = o.spatial_resampling_sample_count;
    r.radius = o.spatial_resampling_radius;
    r.sky = f3{o.sky_color.x, o.sky_color.y, o.sky_color.z};
    return r;
}

// RIS over the emissive triangles: generate_candidate (10_restir_di.cu:78-111) and 09_ris.cu:66-100.
// Randoms are drawn left to right: light pick, two barycentric randoms, then the reservoir's u.
// One candidate: Reservoir::update (reservoir.hpp:22-29) with weight p_hat / light_pdf
CRT_HD void ris_apply_pdf(const Surf& surf, const LightSample& ls, float light_pdf, float u, float p_hat, Res& r)
{
    const float weight = p_hat / light_pdf;
    r.w_sum += weight;
    r.M += 1;
    if (u < weight / r.w_sum)
    {
        r.s.hp = ls.p;
        r.s.hn = ls.n;
        r.s.rad = ls.emissive;
        r.s.op = surf.p;
        r.s.on = surf.n;
        r.s.vis = 0;
    }
}
CRT_HD void ris_apply(const Surf& surf, const LightSample& ls, float inv_n, float u, float p_hat, Res& r)
{
    ris_apply_pdf(surf, ls, inv_n * 1.0f / ls.area, u, p_hat, r);  // 1.0f / size * 1.0f / area (10_restir_di.cu:98-99)
}
template <class L>
CRT_HD void ris_update(const Bvh& bvh, const Surf& surf, const LightSample& ls, float inv_n, float u, bool shadowed, Res& r)
{
    const float p_hat = target_function(bvh, surf.p, surf.n, ls.p, ls.n, ls.emissive, shadowed);
    if (L::kHasPdf) ris_apply_pdf(surf, ls, ls.pdf, u, p_hat, r);
    else ris_apply(surf, ls, inv_n, u, p_hat, r);
}
// The four randoms of a candidate do not depend on earlier candidates, so the light records of kRisBatch
// candidates are requested before the first one is used: kRisBatch gathers in flight per thread instead of one
// (the loop was latency-bound on that gather: profiles/r1/source_g_k_generate_candidate.txt, 59 % long-scoreboard).
#ifndef CRT_RIS_BATCH
#define CRT_RIS_BATCH 2
#endif
constexpr int kRisBatch = CRT_RIS_BATCH;
// pair_mask: see LightsTable::fetch; every lane named in it must run this loop with the same `count`
// 09_ris.cu:66-100 with use_shadowed_target_function: every candidate's target function holds a shadow ray
// (reservoir.hpp:42-59).  The `count` walks run as one loop over walk steps: a lane whose ray is decided applies the
// candidate (Reservoir::update) and draws the next one at once, instead of every lane of the warp waiting for the longest
// walk of the same candidate index.  Per lane the candidates, their randoms and their order are unchanged; the target
// function is evaluated in the reference's order ((1/pi * G) * V) * luminance.
template <class L>
CRT_HD Res ris_candidates_shadowed(const Bvh& bvh, const L& lights, const Surf& surf, int count, Pcg& rng)
{
    Res r = empty_res();
    const float inv_n = 1.0f / (float)lights.n;
    int c = 0;
    bool walking = false;
    LightSample ls;
    ls.p = ls.n = ls.emissive = f3{0.0f, 0.0f, 0.0f};
    ls.area = 0.0f;
    float u = 0.0f, inv_pi_g = 0.0f;
    RaySetup ray;
    Walk w;
    WalkStack stack;
    Hit h;
    const RayLoop loop;
    for (;;)
    {
        bool start;
        if (!loop.next(!walking && c < count, walking, start)) break;
        if (start && !walking && c < count)
        {
            const float r0 = rng.next_f();
            const float r1 = rng.next_f();
            const float r2 = rng.next_f();
            u = rng.next_f();
            ls = lights.finish(lights.fetch(r0), r1, r2);
            inv_pi_g = kInvPi * geometry_term(surf.p, surf.n, ls.p, ls.n);
            ray = setup_ray(surf.p + 0.001f * surf.n, ls.p - surf.p, true);  // check_visibility's segment, far end first
            walk_begin(w, ray);
            h.prim = -1;
            h.t = 0.99f;
            h.u = h.v = 0.0f;
            walking = true;
        }
        if (walking)
        {
            const int state = walk_step<true, true>(bvh, w, stack, ray, 0.0f, h, CRT_LANES_WALKING());
            if (state != kWalkContinue)
            {
                const float V = state == kWalkHitAny ? 0.0f : 1.0f;
                if (L::kHasPdf) ris_apply_pdf(surf, ls, ls.pdf, u, inv_pi_g * V * luminance(ls.emissive), r);
                else ris_apply(surf, ls, inv_n, u, inv_pi_g * V * luminance(ls.emissive), r);
                ++c;
                walking = false;
            }
        }
    }
    return r;
}

// DEFERRED SELECTION.  Reservoir::update copies the whole sample (hit position, hit normal, radiance, origin position,
// origin normal: 15 floats) whenever a candidate is accepted — in SIMT code 14 predicated moves per candidate, executed
// whether or not the lane accepts, and 15 registers that live across the loop.  The sample is a pure function of the
// candidate's three randoms (light pick, two barycentric randoms), so the loop only remembers those of the candidate
// accepted last and the sample is built once, after the loop, by the very calls that built it inside (fetch + finish:
// the same record, the same operations, the same bits).
// MEASURED AND REJECTED (profiles/r2/tuning.txt, batch 37; kept behind -DCRT_RIS_DEFERRED): the loop shrinks from 433 to
// 410 SASS instructions per two candidates, bit-identical — and k_candidate_temporal goes from 2.027 to 2.053 ms.  The
// kernel is bound by the L1's wavefronts for the light-record gathers (l1tex at 85 % of peak), not by issue slots: the
// instructions saved were free, the 33rd gather per pixel is not.  (At 4 blocks per SM, which the smaller live set
// allows with 48 bytes of spills: 2.029 ms; with three records in flight: 2.226 ms.)
struct RisPick
{
    float r0, r1, r2;
    bool has;
};
template <class L>
CRT_HD void ris_update_pick(const Bvh& bvh, const Surf& surf, const LightSample& ls, float inv_n, float u, bool shadowed,
                            float r0, float r1, float r2, Res& r, RisPick& pick)
{
    const float p_hat = target_function(bvh, surf.p, surf.n, ls.p, ls.n, ls.emissive, shadowed);
    const float weight = p_hat / (L::kHasPdf ? ls.pdf : inv_n * 1.0f / ls.area);  // ris_apply_pdf / ris_apply
    r.w_sum += weight;
    r.M += 1;
    if (u < weight / r.w_sum)
    {
        pick.r0 = r0;
        pick.r1 = r1;
        pick.r2 = r2;
        pick.has = true;
    }
}
template <class L>
CRT_HD void ris_pick_finish(const L& lights, const Surf& surf, const RisPick& pick, Res& r)
{
    if (!pick.has) return;
    const LightSample ls = lights.finish(lights.fetch(pick.r0, 0u), pick.r1, pick.r2);
    r.s.hp = ls.p;
    r.s.hn = ls.n;
    r.s.rad = ls.emissive;
    r.s.op = surf.p;
    r.s.on = surf.n;
    r.s.vis = 0;
}

template <class L>
CRT_HD Res ris_candidates(const Bvh& bvh, const L& lights, const Surf& surf, int count, bool shadowed, Pcg& rng,
                          unsigned pair_mask = 0u)
{
#if defined(CRT_RAYS_PER_LANE)  // measured and rejected, see RayLoop (bvh.cuh)
    if (shadowed) return ris_candidates_shadowed(bvh, lights, surf, count, rng);
#endif
    Res r = empty_res();
    const float inv_n = 1.0f / (float)lights.n;
    int i = 0;
#if defined(CRT_RIS_DEFERRED)
    RisPick pick{0.0f, 0.0f, 0.0f, false};
    for (; i + kRisBatch <= count; i += kRisBatch)
    {
        typename L::Raw raw[kRisBatch];
        float r0[kRisBatch], r1[kRisBatch], r2[kRisBatch], u[kRisBatch];
#pragma unroll
        for (int b = 0; b < kRisBatch; ++b)
        {
            r0[b] = rng.next_f();
            r1[b] = rng.next_f();
            r2[b] = rng.next_f();
            u[b] = rng.next_f();
            raw[b] = lights.fetch(r0[b], pair_mask);
        }
#pragma unroll
        for (int b = 0; b < kRisBatch; ++b)
            ris_update_pick<L>(bvh, surf, lights.finish(raw[b], r1[b], r2[b]), inv_n, u[b], shadowed, r0[b], r1[b], r2[b], r, pick);
    }
    for (; i < count; ++i)
    {
        const float r0 = rng.next_f();
        const float r1 = rng.next_f();
        const float r2 = rng.next_f();
        const float u = rng.next_f();
        ris_update_pick<L>(bvh, surf, lights.finish(lights.fetch(r0, pair_mask), r1, r2), inv_n, u, shadowed, r0, r1, r2, r, pick);
    }
    ris_pick_finish(lights, surf, pick, r);
    return r;
#else
    for (; i + kRisBatch <= count; i += kRisBatch)
    {
        typename L::Raw raw[kRisBatch];
        float r1[kRisBatch], r2[kRisBatch], u[kRisBatch];
#pragma unroll
        for (int b = 0; b < kRisBatch; ++b)
        {
            const float r0 = rng.next_f();
            r1[b] = rng.next_f();
            r2[b] = rng.next_f();
            u[b] = rng.next_f();
            raw[b] = lights.fetch(r0, pair_mask);
        }
#pragma unroll
        for (int b = 0; b < kRisBatch; ++b) ris_update<L>(bvh, surf, lights.finish(raw[b], r1[b], r2[b]), inv_n, u[b], shadowed, r);
    }
    for (; i < count; ++i)
    {
        const float r0 = rng.next_f();
        const float r1 = rng.next_f();
        const float r2 = rng.next_f();
        const float u = rng.next_f();
        ris_update<L>(bvh, surf, lights.finish(lights.fetch(r0, pair_mask), r1, r2), inv_n, u, shadowed, r);
    }
    return r;
#endif
}

// temporal_resampling body (10_restir_di.cu:172-233): `r` is this frame's reservoir, `prev` last frame's.
template <class M>
CRT_HD bool temporal_merge(const Bvh& bvh, const Surf& surf, f3 eye, const Opt& opt, Res prev, Res& r, Pcg& rng)
{
    const int cap = 20 * opt.ris_count;  // M-cap, :186-188
    prev.M = prev.M < cap ? prev.M : cap;
    float p_hat_y = target_function(bvh, surf.p, surf.n, prev.s.hp, prev.s.hn, prev.s.rad, opt.shadowed);
    if (opt.reuse) p_hat_y *= (prev.s.vis & 1u) ? 1.0f : 0.0f;
    prev.M = f2i_trunc((float)prev.M * rejection_heuristics<M>(r.s, prev.s, eye));  // int *= float, :211-212
    const float weight = p_hat_y * prev.ucw * (float)prev.M;
    const float u = rng.next_f();
    r.w_sum += weight;  // Reservoir::merge, reservoir.hpp:31-37
    r.M += prev.M;
    const bool accepted = u < weight / r.w_sum;
    if (accepted) r.s = prev.s;
    r.ucw = ucw_of(r, target_function(bvh, surf.p, surf.n, r.s.hp, r.s.hn, r.s.rad, opt.shadowed));
    return accepted;  // false: the sample of `r` (this frame's candidate) survived
}

// M of a merged reservoir after the probabilistic rejection (reservoir.hpp:61-87; int *= float, 10_restir_di.cu:211-212, 357-358)
template <class M>
CRT_HD int rejected_m(const Sample& mine, const Sample& theirs, int their_m, f3 eye)
{
    return f2i_trunc((float)their_m * rejection_heuristics<M>(mine, theirs, eye));
}
// one neighbour of spatial_resampling (10_restir_di.cu:340-370); compares against the *running* reservoir
template <class M>
CRT_HD void spatial_merge(const Bvh& bvh, const Surf& surf, f3 eye, const Opt& opt, Res nb, Res& r, Pcg& rng)
{
    float p_hat_y = target_function(bvh, surf.p, surf.n, nb.s.hp, nb.s.hn, nb.s.rad, opt.shadowed);
    if (opt.reuse) p_hat_y *= (nb.s.vis & 1u) ? 1.0f : 0.0f;
    nb.M = f2i_trunc((float)nb.M * rejection_heuristics<M>(r.s, nb.s, eye));
    const float weight = p_hat_y * nb.ucw * (float)nb.M;
    const float u = rng.next_f();  // third random only for neighbours that survive the rejections
    r.w_sum += weight;
    r.M += nb.M;
    if (u < weight / r.w_sum) r.s = nb.s;
}

// ---- unbiased reuse weights (extension: crt_set_reuse_weights, CRT_REUSE_UNBIASED; DESIGN.md section 15).  A merge
// combines domains: the pixel's own reservoir and each accepted neighbour (spatial), or the current reservoir and the
// history (temporal).  A domain's surface is its *pixel's* primary-hit surface, never the sample's stored origin, so its
// confidence c_j = trunc(M_j * heuristics(S_q, S_j)) depends on the neighbour draws and skips alone.  The merge weight
// is p_hat_q(y_j) * ucw_j * c_j (the stored visibility bit multiplies nothing), r.M accumulates sum c_j as before, and
// after the last domain, with y the selected sample,
//   Z = sum_j c_j [p_hat_j(y) > 0],   ucw = p_hat_q(y) > 0 && Z > 0 ? w_sum / (Z p_hat_q(y)) : 0.
// The rejection heuristics of reservoir.hpp:61-87 (rejection_heuristics above), on two pixel surfaces
template <class M>
CRT_HD float surface_heuristics(const Surf& s0, const Surf& s1, f3 eye)
{
    const float d0 = length(s0.p - eye);
    const float d1 = length(s1.p - eye);
    const float diff = (d1 - d0) * (d1 - d0) / d0;
    float w = 1.0f;
    w *= M::exp(-32.0f * diff);
    const float c = dot(s0.n, s1.n);
    w *= M::pow(c > 0.0f ? c : 0.0f, 8.0f);
    return w;
}
// c_j of a domain with M = m whose pixel surface is `theirs` (int *= float, 10_restir_di.cu:211-212)
template <class M>
CRT_HD int confidence(int m, const Surf& mine, const Surf& theirs, f3 eye)
{
    return f2i_trunc((float)m * surface_heuristics<M>(mine, theirs, eye));
}
// [p_hat_j(y) > 0] at surface s; with the shadowed target function its ray is traced only when the unshadowed value is
// positive (((1/pi G) V) lum > 0 exactly when (1/pi G) lum > 0 and V = 1)
CRT_HD bool target_positive(const Bvh& bvh, const Surf& s, const Sample& y, bool shadowed)
{
    if (!(target_function(bvh, s.p, s.n, y.hp, y.hn, y.rad, false) > 0.0f)) return false;
    return !shadowed || check_visibility(bvh, s.p, s.n, y.hp) != 0.0f;
}
// Z after one more domain of confidence c and surface s
CRT_HD int z_of(int z, int c, const Bvh& bvh, const Surf& s, const Sample& y, bool shadowed)
{
    return target_positive(bvh, s, y, shadowed) ? z + c : z;
}
CRT_HD float ucw_unbiased(float w_sum, int z, float p_hat) { return p_hat > 0.0f && z > 0 ? w_sum / ((float)z * p_hat) : 0.0f; }

// temporal_merge with unbiased weights.  Without reprojection the history's pixel is this pixel and its primary-hit
// surface this frame's (deterministic primary rays, static geometry): c_h = trunc(M_h * heuristics(S_q, S_q)), and
// p_hat_h(y) = p_hat_q(y), so Z = c_own + c_h whenever p_hat_q(y) > 0.
template <class M>
CRT_HD bool temporal_merge_unbiased(const Bvh& bvh, const Surf& surf, f3 eye, const Opt& opt, Res prev, Res& r, Pcg& rng)
{
    const int cap = 20 * opt.ris_count;  // M-cap, :186-188
    prev.M = prev.M < cap ? prev.M : cap;
    const float p_hat_y = target_function(bvh, surf.p, surf.n, prev.s.hp, prev.s.hn, prev.s.rad, opt.shadowed);
    const int c_own = r.M;
    prev.M = confidence<M>(prev.M, surf, surf, eye);
    const float weight = p_hat_y * prev.ucw * (float)prev.M;
    const float u = rng.next_f();
    r.w_sum += weight;
    r.M += prev.M;
    const bool accepted = u < weight / r.w_sum;
    if (accepted) r.s = prev.s;
    r.ucw = ucw_unbiased(r.w_sum, c_own + prev.M, target_function(bvh, surf.p, surf.n, r.s.hp, r.s.hn, r.s.rad, opt.shadowed));
    return accepted;
}
// temporal_merge_unbiased with reprojection (DESIGN.md section 15, "Reprojection"): the history's pixel h is the reprojected
// one and its surface S_h = `hsurf` the previous frame's primary hit there (from the previous Visibility record and the
// previous eye).  has_h = false (no history pixel, sky at h, or M_h = 0) gives c_h = 0.  c_h = trunc(min(M_h, cap) *
// heuristics(S_q, S_h)) with this frame's eye, and Z = c_own [p_hat_q(y) > 0] + c_h [p_hat_h(y) > 0].  With S_h = S_q this
// computes temporal_merge_unbiased's bits.
template <class M>
CRT_HD bool temporal_merge_unbiased_reprojected(const Bvh& bvh, const Surf& surf, bool has_h, const Surf& hsurf, f3 eye,
                                                const Opt& opt, Res prev, Res& r, Pcg& rng)
{
    const int cap = 20 * opt.ris_count;  // M-cap, :186-188
    prev.M = prev.M < cap ? prev.M : cap;
    const float p_hat_y = target_function(bvh, surf.p, surf.n, prev.s.hp, prev.s.hn, prev.s.rad, opt.shadowed);
    const int c_own = r.M;
    prev.M = has_h ? confidence<M>(prev.M, surf, hsurf, eye) : 0;
    const float weight = p_hat_y * prev.ucw * (float)prev.M;
    const float u = rng.next_f();
    r.w_sum += weight;
    r.M += prev.M;
    const bool accepted = u < weight / r.w_sum;
    if (accepted) r.s = prev.s;
    const float p_hat = target_function(bvh, surf.p, surf.n, r.s.hp, r.s.hn, r.s.rad, opt.shadowed);
    int z = c_own;  // ucw_unbiased reads p_hat_q(y) > 0 itself
    if (p_hat > 0.0f && prev.M > 0) z = z_of(z, prev.M, bvh, hsurf, r.s, opt.shadowed);
    r.ucw = ucw_unbiased(r.w_sum, z, p_hat);
    return accepted;
}
// spatial_merge with unbiased weights: `nsurf` is the neighbour pixel's surface, `nb` its input reservoir
template <class M>
CRT_HD void spatial_merge_unbiased(const Bvh& bvh, const Surf& surf, const Surf& nsurf, f3 eye, const Opt& opt, const Res& nb,
                                   Res& r, Pcg& rng)
{
    const float p_hat_y = target_function(bvh, surf.p, surf.n, nb.s.hp, nb.s.hn, nb.s.rad, opt.shadowed);
    const int c = confidence<M>(nb.M, surf, nsurf, eye);
    const float weight = p_hat_y * nb.ucw * (float)c;
    const float u = rng.next_f();
    r.w_sum += weight;
    r.M += c;
    if (u < weight / r.w_sum) r.s = nb.s;
}

// neighbour pixel of spatial_resampling (10_restir_di.cu:309-313): two randoms, Box-Muller, truncation
template <class M>
CRT_HD void spatial_neighbour(int xi, int yi, float radius, Pcg& rng, int& x, int& y)
{
    const float rv0 = rng.next_f();
    const float rv1 = rng.next_f();
    const f2 g = sample_2d_gaussian<M>(rv0, rv1);
    x = f2i_trunc((float)xi + radius / 1.96f * g.x);
    y = f2i_trunc((float)yi + radius / 1.96f * g.y);
}

// resolve (10_restir_di.cu:431-447)
CRT_HD f3 resolve_radiance(const Bvh& bvh, const Surf& surf, f3 color, const Res& r)
{
    const f3 brdf = kInvPi * color;
    const float G = geometry_term(surf.p, surf.n, r.s.hp, r.s.hn);
    const float V = check_visibility(bvh, surf.p, surf.n, r.s.hp);
    return brdf * G * V * r.s.rad * r.ucw;
}

// tone mapping (common/kernels/common.cu:19-74)
CRT_HD float aces(float x)
{
    const float a = 2.51f, b = 0.03f, c = 2.43f, d = 0.59f, e = 0.14f;
    return (x * (a * x + b)) / (x * (c * x + d) + e);
}
CRT_HD uint32_t to_u8(float v)
{
    float s = v * 255.0f;
    s = s > 0.0f ? s : 0.0f;  // max(x, 0): NaN -> 0
    s = s < 255.0f ? s : 255.0f;
    return (uint32_t)s;
}
template <class M>
CRT_HD uint32_t tone_map_rgba8(f4 a)
{
    const float gamma = 1.0f / 2.2f;
    const uint32_t r = to_u8(M::pow(aces(a.x / a.w), gamma));
    const uint32_t g = to_u8(M::pow(aces(a.y / a.w), gamma));
    const uint32_t b = to_u8(M::pow(aces(a.z / a.w), gamma));
    return r | (g << 8) | (b << 16) | (255u << 24);
}

// next bounce (e.g. 08_nee.cu:98-106; core.hpp:209-235): tangent from edge v0->v1
template <class M>
CRT_HD f3 bounce_direction(const Surf& surf, const TriRef& tri, Pcg& rng)
{
    const f3 t = normalize(tri.v(1) - tri.v(0));
    const f3 b = normalize(cross(t, surf.n));
    const float r0 = rng.next_f();
    const float r1 = rng.next_f();
    const float r2 = rng.next_f();
    const f3 l = sample_hemisphere<M>(r0, r1, r2);
    return l.x * t + l.y * surf.n + l.z * b;
}
}  // namespace crt
