// bvh.cuh — compressed 8-wide BVH: node format, ray/triangle test and the traversal loop.
//
// Replaces HIPRT's hiprtGeomTraversalClosestCustomStack behind raytrace()/check_visibility()
// (common/raytrace.hpp:18-52; 06_ao_hiprt.cu:13-33).  B200 has no RT cores, so this is a software
// walk: 80-byte nodes holding eight children as 8-bit boxes on a per-node power-of-two grid (the
// node stream for 10 M triangles stays L2-resident: 126 MB L2), children pre-sorted into octant
// slots so that `slot ^ octant` is a front-to-back priority, one (base, bitmask) stack entry per
// tree level, triangles in 48-byte records fetched as 3 x LDG.128.
//
// The tree only culls.  Accept/reject and the t,u,v bits come from ray_triangle(), which is the
// reference's intersect_ray_triangle (common/core.hpp:91-136) operation for operation; ties on t are
// resolved towards the larger primitive id, which is what the reference's own brute-force loop does
// (04_ao.cu:14-24).  Boxes are padded at build time (bvh_build.cuh) by more than the rounding error
// of both that test and the slab arithmetic below, so no hit the exhaustive loop finds is lost.
#pragma once
#include "vecmath.cuh"

namespace crt
{
constexpr int kLeafMaxTris = 3;  // triangles per leaf child (3 x 8 slots = 24 hit-mask bits)
constexpr int kStackSize = 48;   // >= 2 x depth of the wide tree: one node group + one postponed triangle group
                                 // per level (checked at build time, CRT_ESTACK)

// 80 bytes, read as five 16-byte words.
struct alignas(16) WideNode
{
    float px, py, pz;            // grid origin (one cell below the min corner of the node box)
    uint8_t ex, ey, ez;          // biased exponents: cell size on axis a is 2^(e_a - 127)
    uint8_t imask;               // bit s set: slot s is an inner node
    uint32_t child_base;         // first inner child; child in slot s is child_base + popc(imask & ((1<<s)-1))
    uint32_t tri_base;           // first triangle record of this node's leaf children
    uint8_t meta[8];             // 0: empty slot; inner: 0x20 | (24 + slot); leaf: (unary count 1,3,7) << 5 | offset
                                 // from tri_base — so (meta >> 5) << (meta & 31) is the slot's hit-mask contribution
    uint8_t qlo[3][8];           // per axis, per slot: box min in grid cells (rounded down)
    uint8_t qhi[3][8];           // box max in grid cells (rounded up)
};
static_assert(sizeof(WideNode) == 80, "WideNode must be 80 bytes");

// 48 bytes: v0.xyz + primitive id, v1.xyz, v2.xyz (original vertex bits, untouched)
struct alignas(16) WideTri
{
    float v0x, v0y, v0z;
    int32_t prim;
    float v1x, v1y, v1z, pad1;
    float v2x, v2y, v2z, pad2;
};
static_assert(sizeof(WideTri) == 48, "WideTri must be 48 bytes");

struct Bvh
{
    const WideNode* nodes;
    const WideTri* tris;
    float postpone_ratio;  // triangle-postponing threshold of the walk (0 = never postpone), see walk_step
    uint32_t f32_one = 0x3f800000u;  // bits of 1.0f as a *run-time* value: see byte_to_unit_float
};

struct Hit
{
    float t, u, v;
    int prim;  // -1: miss
};

// common/core.hpp:91-136: t from the plane, then the three signed sub-areas; u = area(p,v2,v0)/A,
// v = area(p,v0,v1)/A.  Accepts tmin <= t <= tmax (NaN fails).
CRT_HD bool ray_triangle(f3 ro, f3 rd, float tmin, float tmax, f3 v0, f3 v1, f3 v2, float& t_out, float& u_out,
                         float& v_out)
{
    const f3 e0 = v1 - v0, e1 = v2 - v1, e2 = v0 - v2;
    const f3 n = cross(e0, e1);
    const float t = dot(v0 - ro, n) / dot(n, rd);
    if (!(tmin <= t && t <= tmax)) return false;
    const f3 p = ro + rd * t;
    const float a0 = dot(n, cross(e0, p - v0));
    const float a1 = dot(n, cross(e1, p - v1));
    const float a2 = dot(n, cross(e2, p - v2));
    if (a0 < 0.0f || a1 < 0.0f || a2 < 0.0f) return false;
    const float a = a0 + a1 + a2;
    t_out = t;
    u_out = a2 / a;
    v_out = a0 / a;
    return true;
}

// The accept / reject decision of ray_triangle() alone, with every operation and comparison spelled as one PTX instruction
// without .ftz, so that the answer is the walk's own — bit for bit — in whatever translation unit it is compiled.  The
// per-pixel kernels of the REFERENCE and FAST builds contract a * b + c into FMAs, and the FAST build's -use_fast_math
// implies -ftz=true, under which even __fmul_rn and a < 0.0f flush denormal operands and results to zero (a sub-area of
// -1e-40 would compare as -0 and accept a triangle the walk rejects); the walk's triangle test is neither contracted nor
// flushed (tests/test_gpu_math_modes.py: rays that leave a floor's edge and cross its plane a denormal distance outside).
// Used for OWN-TRIANGLE PRE-TESTS: a per-pixel kernel that emits a shadow ray knows the triangle the ray starts on, and
// in these scenes a third of the rays towards freshly sampled lights point below that triangle's plane (the reference's
// target function takes |cos|, reservoir.hpp:42-59 / core.hpp:287-295, so such lights are legitimate candidates) and are
// stopped by it at t ~ 1e-3.  An any-hit answer is "some triangle accepts": if this one does, the ray is occluded and
// need not be traced.  Measured (profiles/bvh_lab/lab2.cpp, config 5): 30.6 % of the visibility-reuse rays, 34.5 % of
// their node steps; 0.7 % of the resolve rays (not used there).
#if defined(__CUDA_ARCH__) && defined(CRT_FASTMATH_TU)
// -ftz=true (kernels_fast.cu's FAST build): explicit PTX without .ftz.  Only here: in the builds without flushing the
// intrinsics and plain comparisons below compile to the same operations, and the compiler folds the three sign tests
// into one three-way minimum, which it cannot see through inline assembly.
#define CRT_RN_OP(name, ptx)                                    \
    __device__ __forceinline__ float name(float a, float b)    \
    {                                                           \
        float r;                                                \
        asm(ptx " %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));     \
        return r;                                               \
    }
CRT_RN_OP(rn_mul_f, "mul.rn.f32")
CRT_RN_OP(rn_add_f, "add.rn.f32")
CRT_RN_OP(rn_sub_f, "sub.rn.f32")
CRT_RN_OP(rn_div_f, "div.rn.f32")
#undef CRT_RN_OP
// a < b and a <= b, IEEE (false for NaN), denormals compared as they are
#define CRT_RN_CMP(name, ptx)                                                                          \
    __device__ __forceinline__ bool name(float a, float b)                                             \
    {                                                                                                  \
        uint32_t r;                                                                                    \
        asm("{ .reg .pred p; " ptx " p, %1, %2; selp.u32 %0, 1, 0, p; }" : "=r"(r) : "f"(a), "f"(b)); \
        return r != 0u;                                                                                \
    }
CRT_RN_CMP(rn_lt_f, "setp.lt.f32")
CRT_RN_CMP(rn_le_f, "setp.le.f32")
#undef CRT_RN_CMP
#define CRT_RN_MUL(a, b) rn_mul_f(a, b)
#define CRT_RN_ADD(a, b) rn_add_f(a, b)
#define CRT_RN_SUB(a, b) rn_sub_f(a, b)
#define CRT_RN_DIV(a, b) rn_div_f(a, b)
#define CRT_RN_LT(a, b) rn_lt_f(a, b)
#define CRT_RN_LE(a, b) rn_le_f(a, b)
#elif defined(__CUDA_ARCH__)
#define CRT_RN_MUL(a, b) __fmul_rn(a, b)
#define CRT_RN_ADD(a, b) __fadd_rn(a, b)
#define CRT_RN_SUB(a, b) __fsub_rn(a, b)
#define CRT_RN_DIV(a, b) __fdiv_rn(a, b)
#define CRT_RN_LT(a, b) ((a) < (b))
#define CRT_RN_LE(a, b) ((a) <= (b))
#else
#define CRT_RN_MUL(a, b) ((a) * (b))
#define CRT_RN_ADD(a, b) ((a) + (b))
#define CRT_RN_SUB(a, b) ((a) - (b))
#define CRT_RN_DIV(a, b) ((a) / (b))
#define CRT_RN_LT(a, b) ((a) < (b))
#define CRT_RN_LE(a, b) ((a) <= (b))
#endif
CRT_HD f3 rn_sub(f3 a, f3 b) { return {CRT_RN_SUB(a.x, b.x), CRT_RN_SUB(a.y, b.y), CRT_RN_SUB(a.z, b.z)}; }
CRT_HD f3 rn_cross(f3 a, f3 b)
{
    return {CRT_RN_SUB(CRT_RN_MUL(a.y, b.z), CRT_RN_MUL(a.z, b.y)), CRT_RN_SUB(CRT_RN_MUL(a.z, b.x), CRT_RN_MUL(a.x, b.z)),
            CRT_RN_SUB(CRT_RN_MUL(a.x, b.y), CRT_RN_MUL(a.y, b.x))};
}
CRT_HD float rn_dot(f3 a, f3 b) { return CRT_RN_ADD(CRT_RN_ADD(CRT_RN_MUL(a.x, b.x), CRT_RN_MUL(a.y, b.y)), CRT_RN_MUL(a.z, b.z)); }
CRT_HD bool segment_hits_triangle(f3 ro, f3 rd, float tmin, float tmax, f3 v0, f3 v1, f3 v2)
{
    const f3 e0 = rn_sub(v1, v0), e1 = rn_sub(v2, v1), e2 = rn_sub(v0, v2);
    const f3 n = rn_cross(e0, e1);
    const float t = CRT_RN_DIV(rn_dot(rn_sub(v0, ro), n), rn_dot(n, rd));
    if (!(CRT_RN_LE(tmin, t) && CRT_RN_LE(t, tmax))) return false;
    const f3 p{CRT_RN_ADD(ro.x, CRT_RN_MUL(rd.x, t)), CRT_RN_ADD(ro.y, CRT_RN_MUL(rd.y, t)), CRT_RN_ADD(ro.z, CRT_RN_MUL(rd.z, t))};
    const float a0 = rn_dot(n, rn_cross(e0, rn_sub(p, v0)));
    const float a1 = rn_dot(n, rn_cross(e1, rn_sub(p, v1)));
    const float a2 = rn_dot(n, rn_cross(e2, rn_sub(p, v2)));
    return !(CRT_RN_LT(a0, 0.0f) || CRT_RN_LT(a1, 0.0f) || CRT_RN_LT(a2, 0.0f));
}

struct u4 { uint32_t x, y, z, w; };

CRT_HD u4 load_u4(const void* p)
{
#if defined(__CUDA_ARCH__)
    const uint4 v = __ldg((const uint4*)p);
    return {v.x, v.y, v.z, v.w};
#else
    u4 v;
    memcpy(&v, p, 16);
    return v;
#endif
}

// 32 bytes in one request (sm_100: LDG.E.ENL2.256); p must be 32-byte aligned.  For the random 64-byte gathers of
// the reservoir passes this halves the number of L1 tag lookups per record against 128-bit loads.
struct u8w { u4 lo, hi; };
CRT_HD u8w load_u8w(const void* p)
{
#if defined(__CUDA_ARCH__)
    u8w v;
    // L1::no_allocate: these records are gathered once per use — 32 uniformly random light records per pixel out of 56 MB,
    // a neighbour's reservoir head — and never found in the L1 again (hit rate 6 % in k_candidate_temporal); kept out of it
    // they stop evicting what is reused.  Measured at 4K (profiles/r2/tuning.txt, batch 24): k_candidate_temporal 2.265 ->
    // 2.149 ms, k_spatial_fast 0.745 -> 0.721 ms per pass; an L2::128B fetch hint on the same loads changed nothing.
#if defined(CRT_U8W_ALLOC)
    asm("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
#else
    asm("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
#endif
        : "=r"(v.lo.x), "=r"(v.lo.y), "=r"(v.lo.z), "=r"(v.lo.w), "=r"(v.hi.x), "=r"(v.hi.y), "=r"(v.hi.z), "=r"(v.hi.w)
        : "l"(p));
    return v;
#else
    u8w v;
    memcpy(&v, p, 32);
    return v;
#endif
}

// Quantised plane coordinate q (byte K of a word) as the float 1 + q * 2^-16, without an integer-to-float
// conversion and without a bias subtraction: the byte is added, times 128, into the mantissa of 1.0f.
// intersect_node folds the "1 +" and the 2^-16 into the per-node constants.
//
// On the device this is one IDP.4A (dp4a with the byte weights 128 << 8K and the accumulator 1.0f): it runs on the
// FMA pipe, whose other load in the node test is 48 FFMAs at one issue cycle each, while the ALU pipe (two issue
// cycles per warp instruction) already carries the 32 min/max, the compares and the hit-mask assembly.  The earlier
// form — one PRMT per byte — put 48 more instructions on the ALU pipe, which ncu showed at 65 % utilisation against
// 32 % for the FMA pipe (profiles/r1/ncu_m_*; pipe assignment and rates measured with profiles/microbench/pipes.cu:
// PRMT 2.04, IDP.4A 2.03, FFMA 1.08 cycles; PRMT+IDP.4A overlap, IDP.4A+FFMA add up).
// `one` is 0x3f800000 handed in as a run-time value (Bvh::f32_one, a kernel parameter) so that the compiler keeps
// it in a register instead of re-materialising constants around every conversion.
template <int K>
CRT_HD float byte_to_unit_float(uint32_t w, uint32_t one)
{
#if defined(__CUDA_ARCH__)
#if defined(CRT_NODE_PRMT)
    uint32_t d;  // byte dropped into mantissa bits 8..15 by one PRMT: 1 + q * 2^-15 (kPlaneScale below follows)
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(one), "n"(0x7604 | (K << 4)));
    return __uint_as_float(d);
#else
    return __uint_as_float(__dp4a(w, 128u << (8 * K), one));
#endif
#else
#if defined(CRT_NODE_PRMT)
    return u2f(one | (((w >> (8 * K)) & 0xffu) << 8));
#else
    return u2f(one + (((w >> (8 * K)) & 0xffu) << 7));
#endif
#endif
}
#if defined(CRT_NODE_PRMT)
constexpr float kPlaneScale = 32768.0f;
#else
constexpr float kPlaneScale = 65536.0f;
#endif
// The folded form rounds (o - a * kPlaneScale) once, an error of at most cell/256 in space (cell/512 for the PRMT
// form); child boxes are therefore quantised with a margin of kQuantMargin cells on every side (bvh_build.cuh:
// collapse_item), which keeps the slab test conservative by construction.
constexpr float kQuantMargin = 1.0f / 64.0f;

// test-only instrumentation (tests/emu with -DCRT_COUNT): per-thread node / triangle step counters
#if defined(CRT_COUNT) && !defined(__CUDA_ARCH__)
extern thread_local unsigned long long g_count_nodes, g_count_tris;
#define CRT_COUNT_NODE() (++g_count_nodes)
#define CRT_COUNT_TRI() (++g_count_tris)
#else
#define CRT_COUNT_NODE() ((void)0)
#define CRT_COUNT_TRI() ((void)0)
#endif

// ---- traversal building blocks (shared by the per-thread walk below and the persistent-warp kernels)
struct RaySetup
{
    f3 ro, rd;
    float idx, idy, idz;  // reciprocal direction
    uint32_t octinv;      // 7 ^ octant: `slot ^ octinv` is the front-to-back priority of a child slot
    bool nx, ny, nz;
};
// far_first: visit the children nearest to the ray's *end* first (the octant of the reversed direction).  Only an any-hit
// walk may ask for it — hit / no hit does not depend on the visiting order — and shadow rays towards sampled lights do:
// most occluded ones are blocked next to the light (an emissive face seen from behind sits on its own block), measured
// on the config-4/5 scene at 11.4 -> 8.7 node steps and 12.0 -> 9.9 triangle tests per visibility-reuse ray
// (profiles/bvh_lab/lab.cpp).  A closest-hit walk wants the near children first so that t shrinks early.
CRT_HD RaySetup setup_ray(f3 ro, f3 rd, bool far_first = false)
{
    RaySetup r;
    r.ro = ro;
    r.rd = rd;
    // an exactly axis-parallel component becomes +-1e-20 so that the slab arithmetic never sees 0 * inf
    // (the padded boxes make the perturbation harmless)
    const float dx = fabsf(rd.x) > 1e-20f ? rd.x : copysignf(1e-20f, rd.x);
    const float dy = fabsf(rd.y) > 1e-20f ? rd.y : copysignf(1e-20f, rd.y);
    const float dz = fabsf(rd.z) > 1e-20f ? rd.z : copysignf(1e-20f, rd.z);
    r.idx = 1.0f / dx;
    r.idy = 1.0f / dy;
    r.idz = 1.0f / dz;
    r.nx = dx < 0.0f;
    r.ny = dy < 0.0f;
    r.nz = dz < 0.0f;
    r.octinv = 7u ^ ((r.nx ? 1u : 0u) | (r.ny ? 2u : 0u) | (r.nz ? 4u : 0u));
    if (far_first) r.octinv ^= 7u;
    return r;
}

// Intersect the eight child boxes of one node with the ray segment [tmin, tmax].
// Returns the hit mask: bits 24..31 inner children by priority, bits 0..23 triangles of hit leaf children.
CRT_HD uint32_t intersect_node(const Bvh& bvh, uint32_t node_idx, const RaySetup& r, float tmin, float tmax,
                               uint32_t& child_base, uint32_t& tri_base, uint32_t& imask_out)
{
    CRT_COUNT_NODE();
    const char* np = (const char*)(bvh.nodes + node_idx);
    const u4 n0 = load_u4(np), n1 = load_u4(np + 16), n2 = load_u4(np + 32), n3 = load_u4(np + 48),
             n4 = load_u4(np + 64);
    const uint32_t e_imask = n0.w;
    const float sx = u2f((e_imask & 0xffu) << 23), sy = u2f(((e_imask >> 8) & 0xffu) << 23),
                sz = u2f(((e_imask >> 16) & 0xffu) << 23);
    const uint32_t imask = e_imask >> 24;
    // plane at q cells: t = (p + q*cell - ro) / d = q * a + o with a = cell/d, o = (p - ro)/d.  With the byte
    // read as u = 1 + q / kPlaneScale:  t = u * (a * kPlaneScale) + (o - a * kPlaneScale)
    const float ax = sx * r.idx * kPlaneScale, ay = sy * r.idy * kPlaneScale, az = sz * r.idz * kPlaneScale;  // exact scalings
    const float ox = (u2f(n0.x) - r.ro.x) * r.idx - ax, oy = (u2f(n0.y) - r.ro.y) * r.idy - ay,
                oz = (u2f(n0.z) - r.ro.z) * r.idz - az;
    // word layout: n2 = qlo.x[0..3] qlo.x[4..7] qlo.y[0..3] qlo.y[4..7]; n3 = qlo.z.. qhi.x..; n4 = qhi.y.. qhi.z..
    const uint32_t nearx[2] = {r.nx ? n3.z : n2.x, r.nx ? n3.w : n2.y}, farx[2] = {r.nx ? n2.x : n3.z, r.nx ? n2.y : n3.w};
    const uint32_t neary[2] = {r.ny ? n4.x : n2.z, r.ny ? n4.y : n2.w}, fary[2] = {r.ny ? n2.z : n4.x, r.ny ? n2.w : n4.y};
    const uint32_t nearz[2] = {r.nz ? n4.z : n3.x, r.nz ? n4.w : n3.y}, farz[2] = {r.nz ? n3.x : n4.z, r.nz ? n3.y : n4.w};
    // per-slot hit-mask contribution, four slots per word (Ylitie et al. 2017, listing 2): inner children carry
    // 24 + slot in the low five meta bits, which `^ octinv` turns into the front-to-back priority
    const uint32_t octinv4 = r.octinv * 0x01010101u;
    uint32_t bit_index[2], child_bits[2];
#pragma unroll
    for (int w = 0; w < 2; w++)
    {
        const uint32_t meta4 = w ? n1.w : n1.z;
        const uint32_t is_inner4 = (meta4 & (meta4 << 1)) & 0x10101010u;  // bits 3 and 4 both set: index >= 24
        const uint32_t inner_mask4 = (is_inner4 >> 4) * 0xffu;            // 0xff in every inner slot's byte
        bit_index[w] = (meta4 ^ (octinv4 & inner_mask4)) & 0x1f1f1f1fu;
        child_bits[w] = (meta4 >> 5) & 0x07070707u;
    }
    uint32_t hits = 0;
    const uint32_t one = bvh.f32_one;
#if defined(__CUDA_ARCH__) && !defined(CRT_NODE_NO_FFMA2)
    // sm_100 packed FP32: one FFMA2 evaluates the same plane of two slots (fma.rn.f32x2), halving the issue slots of
    // the 48 plane evaluations; the results are the very same fmaf values.  Measured (profiles/r2/tuning.txt, 4K
    // config 5): raycast 1.98 -> 1.85 ms, visibility-reuse rays 1.81 -> 1.73, resolve rays 3.34 -> 3.26
#define CRT_PLANE2(WORD, K, A, O) __ffma2_rn(make_float2(byte_to_unit_float<K>(WORD, one), byte_to_unit_float<K + 1>(WORD, one)), make_float2(A, A), make_float2(O, O))
#define CRT_SLOT_BITS(W, K) (((child_bits[W] >> (8 * (K))) & 0xffu) << ((bit_index[W] >> (8 * (K))) & 0xffu))
#define CRT_SLOT2(W, K)                                                                                                     \
    {                                                                                                                       \
        const float2 nx2 = CRT_PLANE2(nearx[W], K, ax, ox), ny2 = CRT_PLANE2(neary[W], K, ay, oy), nz2 = CRT_PLANE2(nearz[W], K, az, oz); \
        const float2 fx2 = CRT_PLANE2(farx[W], K, ax, ox), fy2 = CRT_PLANE2(fary[W], K, ay, oy), fz2 = CRT_PLANE2(farz[W], K, az, oz);    \
        const float t0a = fmaxf(fmaxf(nx2.x, ny2.x), fmaxf(nz2.x, tmin)), t1a = fminf(fminf(fx2.x, fy2.x), fminf(fz2.x, tmax));  \
        const float t0b = fmaxf(fmaxf(nx2.y, ny2.y), fmaxf(nz2.y, tmin)), t1b = fminf(fminf(fx2.y, fy2.y), fminf(fz2.y, tmax));  \
        hits |= t0a <= t1a ? CRT_SLOT_BITS(W, K) : 0u;                                                                      \
        hits |= t0b <= t1b ? CRT_SLOT_BITS(W, K + 1) : 0u;                                                                  \
    }
    CRT_SLOT2(0, 0) CRT_SLOT2(0, 2) CRT_SLOT2(1, 0) CRT_SLOT2(1, 2)
#undef CRT_SLOT2
#undef CRT_SLOT_BITS
#undef CRT_PLANE2
#else
#define CRT_SLOT(W, K)                                                                                                      \
    {                                                                                                                       \
        const float t0 = fmaxf(fmaxf(fmaf(byte_to_unit_float<K>(nearx[W], one), ax, ox),                                    \
                                     fmaf(byte_to_unit_float<K>(neary[W], one), ay, oy)),                                   \
                               fmaxf(fmaf(byte_to_unit_float<K>(nearz[W], one), az, oz), tmin));                            \
        const float t1 = fminf(fminf(fmaf(byte_to_unit_float<K>(farx[W], one), ax, ox),                                     \
                                     fmaf(byte_to_unit_float<K>(fary[W], one), ay, oy)),                                    \
                               fminf(fmaf(byte_to_unit_float<K>(farz[W], one), az, oz), tmax));                             \
        const uint32_t bits = ((child_bits[W] >> (8 * K)) & 0xffu) << ((bit_index[W] >> (8 * K)) & 0xffu);                  \
        hits |= t0 <= t1 ? bits : 0u; /* an empty slot has meta 0, hence bits 0 */                                          \
    }
    CRT_SLOT(0, 0) CRT_SLOT(0, 1) CRT_SLOT(0, 2) CRT_SLOT(0, 3) CRT_SLOT(1, 0) CRT_SLOT(1, 1) CRT_SLOT(1, 2) CRT_SLOT(1, 3)
#undef CRT_SLOT
#endif
    child_base = n1.x;
    tri_base = n1.y;
    imask_out = imask;
    return hits;
}

// One triangle record against the ray: the reference test, then the tie rule (smaller t, then larger id).
CRT_HD bool intersect_wide_tri(const WideTri* tp, const RaySetup& r, float tmin, Hit& hit)
{
    CRT_COUNT_TRI();
    const char* q = (const char*)tp;
    const u4 a = load_u4(q), b = load_u4(q + 16), c = load_u4(q + 32);
    float t, u, v;
    if (!ray_triangle(r.ro, r.rd, tmin, hit.t, f3{u2f(a.x), u2f(a.y), u2f(a.z)}, f3{u2f(b.x), u2f(b.y), u2f(b.z)},
                      f3{u2f(c.x), u2f(c.y), u2f(c.z)}, t, u, v))
        return false;
    const int prim = (int)a.w;
    if (!(t < hit.t || hit.prim < 0 || prim > hit.prim)) return false;
    hit.t = t;
    hit.u = u;
    hit.v = v;
    hit.prim = prim;
    return true;
}

// ---- the walk as a resumable state machine (one call of walk_step = one outer iteration)
//
// Divergence control, after Ylitie et al. 2017 ("Efficient Incoherent Ray Traversal on GPUs Through
// Compressed Wide BVHs"): a lane that owns triangles while fewer than kPostponeRatio of the warp's walking
// lanes are in the triangle loop pushes its triangle group on the stack and goes on with node steps, so
// the ~100-instruction triangle test and the ~300-instruction node step each run with many lanes instead
// of every lane waiting for the slowest one in every phase.  Any visiting order gives the same result:
// the closest hit is decided by (t, primitive id) alone.
constexpr float kPostponeRatio = 0.25f;  // default of Bvh::postpone_ratio (CRT_POSTPONE overrides)

#if defined(__CUDA_ARCH__)
#define CRT_LANES_HERE() __popc(__activemask())
#define CRT_LANES_WALKING() __popc(__activemask())
#else
// host build (tests/emu): 0 = never postpone, 1 = postpone whenever allowed (exercises that path)
extern int g_emu_postpone;
#define CRT_LANES_HERE() (g_emu_postpone ? 0 : 32)
#define CRT_LANES_WALKING() 32
#endif

// The stack lives in local memory (dynamic indexing); everything else of the walk's state is meant for registers, so
// the two are separate objects: as members of one struct the scalars were written back to local memory after every
// update (23 STL + 10 LDL per node step in k_trace_shadow_queue, profiles/r1).  One 64-bit entry per push / pop.
struct WalkEntry
{
    uint32_t base, mask;
};
struct alignas(8) WalkStack
{
    WalkEntry e[kStackSize];
};
// MEASURED AND REJECTED (kept behind -DCRT_RAYS_PER_LANE; profiles/r2/tuning.txt): 06_ao at 32 rays 17.5 ms per frame with
// the reference's lockstep loop over rays, 23.0 ms with this loop (26.7 ms without the start-together rule); 09_ris with
// the shadowed target 179.7 against 203.2 ms.  The walks of these single-kernel examples are short (a 3 034-triangle
// scene; any-hit rays that stop early), so the two ballots and the re-entered walk_step per iteration cost more than
// the idle lanes they save.
// Per-lane ray loops (px_ao, ris_candidates_shadowed): every lane walks its own sequence of rays, one walk step per
// iteration, and draws its next ray when the current one is decided — instead of all lanes waiting for the warp's longest
// walk of the same ray index.  Two things keep that efficient: the lanes that entered the loop together stay together
// until the last one is finished (the ballots name the entry mask, so every iteration reconverges there), and a lane
// waits for its next ray until at least kStartTogether lanes wait with it or nobody walks any more, so that ray set-up
// (sampling, IEEE divisions, sinf / cosf) runs with many lanes.  (Starting each lane's ray the moment it was free made
// 06_ao at 32 rays 17.4 -> 26.7 ms per frame: the set-up then ran in almost every iteration for one or two lanes.)
constexpr int kStartTogether = 8;
struct RayLoop
{
#if defined(__CUDA_ARCH__)
    unsigned mask;
    __device__ __forceinline__ RayLoop() : mask(__activemask()) {}
    // false: every lane of the loop is finished.  start: lanes that want a ray may set it up in this iteration.
    __device__ __forceinline__ bool next(bool wants_a_ray, bool walking, bool& start) const
    {
        const unsigned w = __ballot_sync(mask, wants_a_ray), b = __ballot_sync(mask, walking);
        start = __popc(w) >= kStartTogether || b == 0u;
        return (w | b) != 0u;
    }
#else
    bool next(bool wants_a_ray, bool walking, bool& start) const
    {
        start = true;
        return wants_a_ray || walking;
    }
#endif
};

struct Walk
{
    int sp;
    uint32_t ng_base, ng_mask;  // node group: inner-child hits in bits 24..31 (by priority), imask in bits 0..7
    uint32_t tri_base, tmask;   // triangle group: hit triangles of the last node's leaf children
};
CRT_HD void walk_begin(Walk& w, const RaySetup& r)
{
    w.sp = 0;
    // the root as the only child (slot 0) of a virtual group at base 0
    w.ng_base = 0;
    w.ng_mask = 1u << (24 + (0u ^ r.octinv));
    w.tri_base = 0;
    w.tmask = 0;
}
enum { kWalkContinue = 0, kWalkDone = 1, kWalkHitAny = 2 };

// lanes_walking: number of lanes of the warp that entered this iteration (read at a converged point)
template <bool ANY, bool POSTPONE>
CRT_HD int walk_step(const Bvh& bvh, Walk& w, WalkStack& st, const RaySetup& r, float tmin, Hit& hit, int lanes_walking)
{
    // ---- node work: at most one node step
    if (w.tmask == 0)
    {
        if ((w.ng_mask >> 24) == 0)
        {
            if (w.sp == 0) return kWalkDone;
            --w.sp;
            const WalkEntry top = st.e[w.sp];
            const uint32_t b = top.base, m = top.mask;
            if (m >> 24)
            {
                w.ng_base = b;
                w.ng_mask = m;
            }
            else  // a postponed triangle group
            {
                w.tri_base = b;
                w.tmask = m;
            }
        }
        if (w.tmask == 0)
        {
            const int bit = 31 - clz32(w.ng_mask);  // bits 24..31 are non-empty here
            w.ng_mask &= ~(1u << bit);
            const uint32_t slot = (uint32_t)(bit - 24) ^ r.octinv;
            const uint32_t node_idx = w.ng_base + (uint32_t)popc(w.ng_mask & 0xffu & ((1u << slot) - 1u));
            if (w.ng_mask >> 24)
            {
                st.e[w.sp] = WalkEntry{w.ng_base, w.ng_mask};
                ++w.sp;
            }
            uint32_t imask;
            const uint32_t hits = intersect_node(bvh, node_idx, r, tmin, hit.t, w.ng_base, w.tri_base, imask);
            w.ng_mask = (hits & 0xff000000u) | imask;
            w.tmask = hits & 0x00ffffffu;
        }
    }
    // ---- triangle work
    const WideTri* tp = bvh.tris + w.tri_base;
#if defined(__CUDA_ARCH__) && defined(CRT_POSTPONE_BALLOT)
    // experiment: decide once per step, from a ballot at the point where the node work has rejoined, how many of the
    // warp's walking lanes own triangles — instead of counting the lanes that happen to execute the loop head together
    const unsigned walking_now = __activemask();
    const int lanes_with_tris = __popc(__ballot_sync(walking_now, w.tmask != 0u));
    if (POSTPONE && w.tmask && (w.ng_mask >> 24) != 0 && (float)lanes_with_tris < bvh.postpone_ratio * (float)__popc(walking_now))
    {
        st.e[w.sp] = WalkEntry{w.tri_base, w.tmask};
        ++w.sp;
        w.tmask = 0;
    }
#endif
    while (w.tmask)
    {
#if !defined(CRT_POSTPONE_BALLOT)
        if (POSTPONE && (w.ng_mask >> 24) != 0 && (float)CRT_LANES_HERE() < bvh.postpone_ratio * (float)lanes_walking)
#else
        if (false)
#endif
        {
            st.e[w.sp] = WalkEntry{w.tri_base, w.tmask};
            ++w.sp;
            w.tmask = 0;
            break;
        }
        const int i = 31 - clz32(w.tmask & (0u - w.tmask));
        w.tmask &= w.tmask - 1u;
        if (intersect_wide_tri(tp + i, r, tmin, hit) && ANY) return kWalkHitAny;
    }
    return kWalkContinue;
}

// Closest hit (ANY = false) in [tmin, tmax]: smallest t, ties -> larger primitive id.
// Any hit (ANY = true): returns at the first accepted triangle; only hit.prim >= 0 is meaningful.
// FAR_FIRST (any-hit only): see setup_ray.
// trace_seeded: the same walk started from a hit the caller already holds (hit.prim >= 0, hit.t its distance; or
// hit.prim = -1 and hit.t = tmax for none).  The walk culls with hit.t from its first node on and replaces the seed by
// any triangle that beats it under the tie rule, so the result is the unseeded walk's as long as the seed is what
// ray_triangle() returns for a triangle of this tree (when the walk meets that triangle again it computes the same t and
// the same id, which replaces nothing).
template <bool ANY, bool FAR_FIRST = false>
CRT_HD bool trace_seeded(const Bvh& bvh, f3 ro, f3 rd, float tmin, Hit& hit)
{
    static_assert(ANY || !FAR_FIRST, "a closest-hit walk visits near children first");
    const RaySetup r = setup_ray(ro, rd, FAR_FIRST);
#if !defined(CRT_WALK_SPLIT_OBJECTS)
    // Stack and scalars as members of one object: the compiler then keeps the scalars in local memory too — more
    // instructions, and yet faster here: this per-thread walk's divergence control (triangle postponing by
    // __activemask() counts) depends on where the compiler lets the lanes rejoin, and with register-resident scalars it
    // rejoined less (k_raycast 26.6 -> 24.7 lanes per instruction, 1.98 -> 2.11 ms; 08_nee 3.9 -> 4.6 ms per frame:
    // profiles/r2/tuning.txt).  The persistent shadow-ray kernel has no such dependence and uses the split objects.
    struct
    {
        WalkStack stack;
        Walk w;
    } both;
    Walk& w = both.w;
    WalkStack& stack = both.stack;
#else
    Walk w;
    WalkStack stack;
#endif
    walk_begin(w, r);
    for (;;)
    {
        const int lanes = CRT_LANES_WALKING();
        const int state = walk_step<ANY, true>(bvh, w, stack, r, tmin, hit, lanes);
        if (state != kWalkContinue) break;
    }
    return hit.prim >= 0;
}
template <bool ANY, bool FAR_FIRST = false>
CRT_HD bool trace(const Bvh& bvh, f3 ro, f3 rd, float tmin, float tmax, Hit& hit)
{
    hit.prim = -1;
    hit.t = tmax;
    hit.u = hit.v = 0.0f;
    return trace_seeded<ANY, FAR_FIRST>(bvh, ro, rd, tmin, hit);
}
}  // namespace crt
