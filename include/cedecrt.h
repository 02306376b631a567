/* cedecrt.h — C ABI of libcedecrt.so: the B200 (sm_100a) drop-in for the ReSTIR DI hot path of
 * yumcyaWiz/CEDEC-2024-RT (examples 06-10).
 *
 * Every entry point names the reference interface it replaces (paths relative to the reference
 * repository).  All functions return 0 on success or a CRT_E* code; nothing throws, nothing traps
 * (the reference ignores Orochi return codes or SIGTRAPs through SH_ASSERT, common/shader.hpp:10-16).
 * There is no CPU fallback: without a CUDA device crt_init() fails with CRT_ENODEVICE.
 *
 * Struct layouts are the reference's, byte for byte (static_asserts in csrc/api.cu):
 *   crt_triangle     common/core.hpp:38-43        60 B
 *   crt_visibility   common/core.hpp:167-172      16 B
 *   crt_reservoir    common/reservoir.hpp:5-38    76 B (sample 64 B)
 *   crt_options      common/options.hpp:4-23      48 B
 *   crt_raygen       common/camera.hpp:5-9        36 B
 *   crt_buffer       common/typedbuffer.hpp:14-20 16 B  {T* data; size_t size:63, isDevice:1}
 */
#ifndef CEDECRT_H
#define CEDECRT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct { float x, y, z; } crt_float3;
typedef struct { float x, y, z, w; } crt_float4;

typedef struct { crt_float3 vertices[3]; crt_float3 color; crt_float3 emissive; } crt_triangle;
typedef struct { float uv[2]; int32_t index; int32_t _pad; } crt_visibility;
typedef struct
{
    crt_float3 origin_position, origin_normal, hit_position, hit_normal, radiance;
    uint8_t visibility; /* C++ bool */
    uint8_t _pad[3];
} crt_reservoir_sample;
typedef struct { crt_reservoir_sample sample; float w_sum; float ucw; int32_t M; } crt_reservoir;
typedef struct
{
    uint8_t accumulate; uint8_t _p0[3];
    int32_t max_depth;
    crt_float3 sky_color;
    int32_t ris_sample_count;
    float rejection_heuristics_threshold; /* never read by any kernel, as in the reference */
    uint8_t use_temporal_resampling;
    uint8_t use_spatial_resampling; uint8_t _p1[2];
    int32_t spatial_resampling_sample_count;
    float spatial_resampling_radius;
    int32_t spatial_resampling_passes; /* host-side loop count */
    uint8_t use_shadowed_target_function;
    uint8_t use_visibility_reuse; uint8_t _p2[2];
} crt_options;
typedef struct { crt_float3 m_origin, m_right, m_up; } crt_raygen;

/* Device view of TypedBuffer<T> exactly as the reference passes it to kernels (ShaderArgument::ptr,
 * common/shader.hpp:50-54,82-83): 16 bytes by value.  `size` counts elements; bit 63 is m_isDevice. */
typedef struct { void* data; uint64_t size_and_flag; } crt_buffer;
#define CRT_BUFFER_SIZE(b) ((b).size_and_flag & 0x7fffffffffffffffull)

typedef struct crt_ctx crt_ctx;              /* one per GPU: device + stream (10_restir_di.cpp:30-53) */
typedef struct crt_geometry_t* crt_geometry; /* opaque 8-byte handle in hiprtGeometry's argument slot */

enum
{
    CRT_OK = 0,
    CRT_ENODEVICE = 1, /* no CUDA device / driver: the library never computes on the CPU */
    CRT_ECUDA = 2,     /* a CUDA runtime call failed; see crt_last_error() */
    CRT_EINVAL = 3,    /* bad argument (null pointer, size mismatch, unknown kernel name) */
    CRT_ENOMEM = 4,
    CRT_ESTACK = 5     /* BVH deeper than the traversal stack */
};

/* arithmetic of the per-pixel kernels (Box-Muller log/sin/cos of the neighbour draw, exp/pow of the rejection
 * heuristics, pow in tone mapping and AO, and whether a*b+c is contracted).  Ray traversal and the triangle test are
 * outside all of this: they run the reference's test operation for operation in every mode, so primitive ids and
 * hit/no-hit never depend on the mode.
 *   CRT_MATH_REFERENCE  fused frame: FMA contraction, IEEE division and square root, CUDA's libdevice functions —
 *                       nvcc's and NVRTC's defaults, i.e. the arithmetic of the reference's own GPU build
 *                       (10_restir_di.cpp:56-70 passes no floating-point option).  Default.  The per-kernel entry
 *                       points treat it as LIBDEVICE.  Against the CPU oracle: radiance inside the north star's
 *                       tolerance (mean relative L1 <= 1e-3 after 64 frames; tests/test_gpu_parity.py).
 *   CRT_MATH_LIBDEVICE  libdevice functions with every + - * / rounded once in source order (no contraction): the
 *                       CPU oracle's own arithmetic up to the last ulp of its libm calls.
 *   CRT_MATH_EXACT      as LIBDEVICE with correctly rounded transcendentals (via double); bit-identical to the CPU
 *                       oracle's mode 1 — the mode of every bit-exact parity test.
 *   CRT_MATH_FAST       fused frame only (the per-kernel entry points treat it as LIBDEVICE): the reservoir kernels
 *                       (candidates + temporal, spatial passes, resolve's shading) run with FMA contraction, approximate
 *                       division / square root and the hardware exp2/log2/sin/cos approximations.  Rays are still
 *                       traced and triangles tested with the exact arithmetic, so primitive ids are unaffected; radiance
 *                       stays inside the north star's tolerance (mean relative L1 <= 1e-3 after 64 frames, measured
 *                       ~1e-5: tests/test_gpu_parity.py) but is no longer bit-comparable with the oracle. */
enum { CRT_MATH_LIBDEVICE = 0, CRT_MATH_EXACT = 1, CRT_MATH_FAST = 2, CRT_MATH_REFERENCE = 3 };

/* ---- context, memory, timing ------------------------------------------------------------------ */
/* replaces oroInitialize/oroInit/oroDeviceGet/oroCtxCreate/oroStreamCreate (10_restir_di.cpp:30-53) */
int crt_init(int device, crt_ctx** out);
int crt_shutdown(crt_ctx* ctx);
const char* crt_device_name(crt_ctx* ctx);  /* oroGetDeviceProperties().name (10_restir_di.cpp:47-52) */
const char* crt_last_error(void);
int crt_set_math_mode(crt_ctx* ctx, int mode);
/* Light selection (extension; the reference always selects uniformly).  Applies to every kernel that samples a light:
 * the candidates of 10_restir_di (crt_generate_candidate, the fused frame), the NEE sample of crt_path_trace_08 and the
 * candidates of crt_path_trace_09.
 *   CRT_LIGHTS_UNIFORM  one emissive triangle in n, pdf 1/n * 1/area: the reference's behaviour.  Default.
 *   CRT_LIGHTS_POWER    in proportion to emitted power P_i = max(0, luminance(Le_i)) * area_i, with every light keeping a
 *                       nonzero probability (so RIS stays unbiased against the reference's target function): light i owns
 *                       c_i >= 1 of K = 2^log2_slots slots, K >= n, and is selected with probability c_i / K.  The K - n
 *                       slots beyond one per light go by power, so the mix is about (n / K) uniform.  log2_slots = 0
 *                       picks min(23, ceil(log2 n) + 2) (about 1/4 uniform, 3/4 by power).  The table holds one
 *                       64-byte record per slot (K * 64 bytes per geometry).  A log2_slots with 2^k < n or k > 23, or
 *                       more than 2^23 lights, makes the first call that samples lights return CRT_EINVAL.
 * Temporal and spatial resampling, resolve and the shadow rays do not read the source pdf and are unchanged.  The table
 * is a pure function of the triangles and the light list (built in integers from quantised powers), so every row slab
 * and every GPU builds the same one.  It is cached per (geometry, light list pointer, count, mode, K) and rebuilt after
 * crt_refit_geometry; a host that changes emission in place calls crt_lights_changed (power mode reads Ke for its slot
 * counts, and the records of both modes hold a copy of Ke). */
enum { CRT_LIGHTS_UNIFORM = 0, CRT_LIGHTS_POWER = 1 };
int crt_set_light_sampling(crt_ctx* ctx, int mode, int log2_slots);
/* the light records the context's kernels would read for this light list (built now if needed), for inspection: K
 * LightRec records of 16 floats {v0.xyz, pdf, v1.xyz, n.x, v2.xyz, n.y, Le.xyz, n.z} with pdf = sel * 1 / area
 * (sel = c_i / K in power mode, 1 / n in uniform mode, where *n_slots = n); device memory owned by the geometry,
 * valid until the next rebuild */
int crt_light_sampling_table(crt_ctx* ctx, crt_geometry geom, crt_buffer lights, const void** d_records, uint32_t* n_slots);
/* the host has changed emission (Ke) of triangles in place: the light records are rebuilt at their next use */
int crt_lights_changed(crt_ctx* ctx, crt_geometry geom);
/* Presampled light tiles (extension; RTXDI's light presampling).  Off by default (log2_tiles = log2_tile_size = 0).
 * Applies only to the light pick of 10_restir_di's candidates: crt_generate_candidate (directly and through crt_launch),
 * the fused frame's candidate + temporal kernel and the per-kernel path crt_restir_di_frame falls back to.  The NEE
 * sample of crt_path_trace_08 and the candidates of crt_path_trace_09 keep reading the source records.
 * Once per frame the context draws T = 2^log2_tiles tiles of S = 2^log2_tile_size records from the source records the
 * candidates read otherwise (one per light, or the K slots of CRT_LIGHTS_POWER): entry e of tile t copies source slot
 * (uint32)(u * (float)K), u a PCG draw keyed on (frame, t, e) only, pdf included.  The pixel (xi, yi) draws its candidates
 * from tile hash(frame, xi >> 3, yi >> 2) & (T - 1) with nth = (uint32)(rv0 * (float)S), in global pixel coordinates, so
 * every row range agrees; it consumes the same random numbers as without tiles.  Each candidate keeps the source's
 * marginal distribution and divides by the record's own pdf, so RIS stays unbiased; candidates that share a tile are
 * correlated, which costs variance, not bias.  Reuse, resolve and the shadow rays are unchanged.  The candidates then
 * read T * S * 64 bytes per frame whatever the light count.  log2_tiles and log2_tile_size are in [0, 16] with
 * log2_tiles + log2_tile_size <= 22; anything else returns CRT_EINVAL.  The tiles are owned by the context, rebuilt on its
 * stream when the frame, the source records, T or S change. */
int crt_set_light_tiles(crt_ctx* ctx, int log2_tiles, int log2_tile_size);
/* the tiles of `frame` the candidates would read for this light list (built now if needed), for inspection: *n_tiles *
 * *tile_size LightRec records (crt_light_sampling_table's layout), tile t first at record t * *tile_size; device memory
 * owned by the context, valid until the next rebuild.  CRT_EINVAL while tiles are off. */
int crt_light_tiles(crt_ctx* ctx, crt_geometry geom, crt_buffer lights, int frame, const void** d_records, uint32_t* n_tiles,
                    uint32_t* tile_size);
/* Reuse weights (extension; the reference's reuse is biased).  Applies to every kernel that merges reservoirs:
 * crt_temporal_resampling and crt_spatial_resampling (directly and through crt_launch), the fused frame's candidate +
 * temporal kernel and crt_restir_spatial_pass, and the per-kernel path crt_restir_di_frame falls back to.
 *   CRT_REUSE_REFERENCE  the reference's merge: a neighbour's M counts whether or not it could have produced the selected
 *                        sample, ucw = w_sum / (M p_hat), the rejection heuristics compare the running reservoir's sample
 *                        origin, and with use_visibility_reuse the stored visibility bit zeroes a weight.  Default.
 *   CRT_REUSE_UNBIASED   1/Z weights.  A merge combines domains: the pixel's own input reservoir and each accepted
 *                        neighbour (spatial), or the current reservoir and the history (temporal).  A domain's surface
 *                        is its pixel's primary-hit surface (position and shading normal), not the sample's origin.
 *                        Which neighbours are visited is exactly the reference's (the same draws, skips and random
 *                        stream).  Domain j has confidence c_j = trunc(M_j * rejection_heuristics(S_q, S_j)) — the
 *                        reference's formula on the two pixel surfaces; the temporal M cap 20 * ris_sample_count applies
 *                        first — and its sample y_j merges with weight p_hat_q(y_j) * ucw_j * c_j; the visibility bit
 *                        weighs nothing (use_visibility_reuse still traces and stores it, and resolve still reads it to
 *                        skip a shadow ray).  Selection is unchanged and M accumulates sum c_j.  After the last domain,
 *                        for the selected sample y:
 *                          Z = sum over domains j (the pixel's own, c = its input M, included) of c_j [p_hat_j(y) > 0]
 *                          ucw = p_hat_q(y) > 0 && Z > 0 ? w_sum / (Z p_hat_q(y)) : 0
 *                        with p_hat_j the reference's target function at domain j's surface (including a shadow ray
 *                        under use_shadowed_target_function, traced only when the unshadowed value is positive).
 *                        Candidate generation is a single domain and unchanged.  Without reprojection the history's
 *                        surface is the pixel's own, so temporal Z = M whenever p_hat_q(y) > 0.  After
 *                        crt_refit_geometry, without the previous frame's triangles (crt_temporal_resampling_reprojected_motion,
 *                        crt_restir_set_previous_triangles; DESIGN.md section 17) the history is merged from where the
 *                        moved surface point now lies, and S_h is rebuilt on this frame's triangles: that changes which
 *                        history is merged and its c_h, not the estimator's unbiasedness, because the target function's
 *                        support does not depend on S_h's orientation.  Under use_shadowed_target_function, where p_hat
 *                        includes visibility, neither form is claimed unbiased across a refit.
 * CRT_REUSE_UNBIASED is refused (CRT_EINVAL) with a previous camera that comes without the previous frame's surfaces
 * (crt_temporal_resampling_reprojected, and a camera set with crt_restir_set_previous_camera: use
 * crt_temporal_resampling_reprojected_surfaces and crt_restir_set_previous_frame) and in the fused frame on a row range
 * narrower than the image or with slab links, unless crt_restir_set_halo_surfaces is on (otherwise the G-buffer of halo
 * rows is not kept); the per-kernel path takes row ranges.  An unknown mode is CRT_EINVAL. */
enum { CRT_REUSE_REFERENCE = 0, CRT_REUSE_UNBIASED = 1 };
int crt_set_reuse_weights(crt_ctx* ctx, int mode);
/* Multi-GPU row slabs: the kernels of this context compute only image rows yi in [y_begin, y_end) (y_end < 0:
 * to the image height).  Pixel coordinates, RNG keys and buffer indices stay global, so N slabs give exactly
 * the single-GPU frame; buffers are full-size and the host exchanges the halo rows the spatial pass reads. */
int crt_set_row_range(crt_ctx* ctx, int y_begin, int y_end);
/* Frame overlap (off by default; the reference's loop is strictly serial).  With it on, crt_restir_frame_end issues the
 * tail of the fused frame — the resolve rays and tone mapping, which touch only their own ray queue, `accumulation` and
 * `pixels` — to a second stream of the context, so the next frame's crt_restir_frame_begin / spatial passes run beside
 * it and fill the drain of the persistent ray kernel (and the other way round): same images, frames still complete in
 * order.  Every entry point that reads or writes `accumulation` / `pixels`, copies memory, synchronises or times
 * (crt_restir_frame_end itself, crt_tone_mapping, crt_clear, crt_resolve, crt_memcpy_*, crt_sync, crt_timer_*, ...)
 * first orders the context's stream after the tail in flight; a host that reads those buffers with its own stream
 * operations calls crt_frame_join first, or orders its copy after crt_get_tail_stream()'s work to keep the overlap. */
int crt_set_frame_overlap(crt_ctx* ctx, int on);
/* With overlap on: trace the primary rays of the NEXT frame now, on a third stream and into a Visibility buffer of the
 * context's own, beside the kernels of the frame in flight (raycast, 10_restir_di.cu:9-34, needs nothing but the camera
 * and the geometry).  The next crt_restir_frame_begin / crt_restir_di_frame that arrives with exactly this camera,
 * geometry, image size and row range copies those rows into its `visibility` buffer instead of tracing them; any other
 * call traces as usual and the prefetch is dropped.  A no-op while overlap is off. */
int crt_restir_prefetch_raycast(crt_ctx* ctx, int width, int height, crt_geometry geom, crt_raygen next_raygen);
int crt_frame_join(crt_ctx* ctx);
void* crt_get_tail_stream(crt_ctx* ctx); /* NULL until overlap has been switched on once */
/* use an existing CUDA stream (e.g. torch's) instead of the context's own; NULL restores it */
int crt_set_stream(crt_ctx* ctx, void* cuda_stream);
void* crt_get_stream(crt_ctx* ctx);
/* number of CUDA kernels this context has launched so far (bench.py reports it as gpu_launches) */
unsigned long long crt_launch_count(crt_ctx* ctx);
/* shadow rays (check_visibility, raytrace.hpp:45-52) traced through the wavefront queue since crt_init — out[0]
 * visibility-reuse rays (10_restir_di.cu:127-131), out[1] resolve rays (:443-444); waits for the stream.  The fused frame traces fewer than the reference's two per diffuse pixel: the visibility-reuse ray
 * only for candidates that survive the temporal merge, the resolve ray only when it has not been traced before. */
int crt_shadow_rays_traced(crt_ctx* ctx, unsigned long long out[2]);
/* rays traced inside the single-kernel examples (crt_ao_06, crt_path_trace_07/08/09) since crt_init — out[0]
 * closest-hit rays (camera and bounce rays), out[1] shadow / AO rays, counted per path vertex as SURVEY.md section 8d
 * counts them (08_nee.cu:43,76-77; 09_ris.cu:90-93,112,116-119; 06_ao_hiprt.cu:71-82); waits for the stream */
int crt_inline_rays_traced(crt_ctx* ctx, unsigned long long out[2]);
/* shadow rays that needed no walk since crt_init: the per-pixel kernel that emits a ray tests it against the triangle it
 * starts on (the reference's own intersect_ray_triangle, core.hpp:91-136, on the segment of check_visibility,
 * raytrace.hpp:45-52); a hit there is the walk's answer "occluded".  out[0]: visibility-reuse rays of 10_restir_di
 * (generate_candidate, 10_restir_di.cu:127-131), out[1]: shadow rays of the wavefront 08_nee / 09_ris.  These rays are
 * not in crt_shadow_rays_traced / crt_inline_rays_traced; traced + decided = the rays the reference traces. */
int crt_rays_decided_at_emission(crt_ctx* ctx, unsigned long long out[2]);
/* TypedBuffer<T>(DEVICE).allocate / dtor / toDevice / toHost (common/typedbuffer.hpp:29-77);
 * memory is uninitialised, as with oroMalloc */
int crt_malloc(crt_ctx* ctx, size_t bytes, void** out);
int crt_free(crt_ctx* ctx, void* p);
int crt_memset(crt_ctx* ctx, void* p, int byte, size_t bytes);
int crt_memcpy_h2d(crt_ctx* ctx, void* dst, const void* src, size_t bytes);       /* oroMemcpyHtoD */
int crt_memcpy_d2h(crt_ctx* ctx, void* dst, const void* src, size_t bytes);       /* oroMemcpyDtoH */
/* device to device on the context's stream, asynchronous (extension: a host keeping last frame's triangle array) */
int crt_memcpy_d2d(crt_ctx* ctx, void* dst, const void* src, size_t bytes);
int crt_memcpy_d2h_async(crt_ctx* ctx, void* dst, const void* src, size_t bytes); /* oroMemcpyDtoHAsync, :386 */
int crt_sync(crt_ctx* ctx);                                                       /* oroStreamSynchronize, :389 */
/* OroStopwatch (libs/orochi/Orochi/OrochiUtils.h:179-209): events on the context's stream */
int crt_timer_start(crt_ctx* ctx);
int crt_timer_stop_ms(crt_ctx* ctx, float* ms);

/* per-kernel device times (the breakdown behind the reference's single on-screen "kernel: x ms",
 * 10_restir_di.cpp:382-383,410): between begin and end every kernel launched through this context is followed by
 * an event; end synchronises and returns, per launch in order, a name ('\n'-separated) and the milliseconds
 * since the previous launch finished */
int crt_profile_begin(crt_ctx* ctx);
int crt_profile_end(crt_ctx* ctx, char* names, size_t names_cap, float* ms, int ms_cap, int* count);

/* RayGenerator::lookat (common/camera.hpp:11-25), evaluated on the host like the reference does */
void crt_raygen_lookat(crt_raygen* rg, const float eye[3], const float center[3], const float up[3], float fovy,
                       int width, int height);

/* ---- geometry: replaces hiprtCreateContext + buildHiprtGeometry (10_restir_di.cpp:74-79,220;
 * common/loader.hpp:68-112).  `triangles` is a DEVICE pointer to n reference Triangle structs; the
 * BVH (compressed 8-wide nodes) is built on the GPU, synchronously.  The handle is passed by value
 * to the kernels in hiprtGeometry's slot. */
int crt_build_geometry(crt_ctx* ctx, const crt_triangle* d_triangles, size_t n, crt_geometry* out);
int crt_destroy_geometry(crt_ctx* ctx, crt_geometry g);
/* The host has moved vertices in the triangle array the tree was built over (same count, same order): bring the tree
 * up to date without rebuilding it — HIPRT's hiprtBuildOperationUpdate (libs/hiprt/hiprt/hiprt_types.h:131-135), which
 * the reference never calls (it builds once, loader.hpp:106-110).  Topology is kept, boxes are recomputed bottom-up;
 * hits stay exact (the tree only culls).  Synchronous.  With frame overlap it first orders itself after the frame tail
 * and the primary-ray prefetch in flight, which walk the tree; a host that writes the vertices on a stream of its own calls
 * crt_frame_join first, since the tail may still read them. */
int crt_refit_geometry(crt_ctx* ctx, crt_geometry g);
/* statistics: {n_tris, n_wide_nodes, max_depth, build_ms, node_bytes, tri_bytes, box padding, last refit_ms} */
int crt_geometry_stats(crt_geometry g, double out[8]);
/* single-ray probes for tests (device arrays of n rays: origin, direction as float3, tmin/tmax);
 * closest: out_prim (-1 = miss), out_tuv (t,u,v) — tie rule: smallest t, then largest primitive id
 * (examples/04_ao/04_ao.cu:14-24).  any: out_prim = 1 if any hit in [tmin,tmax] else 0. */
int crt_trace_closest(crt_ctx* ctx, crt_geometry g, size_t n, const float* d_org, const float* d_dir, float tmin,
                      float tmax, int32_t* d_out_prim, float* d_out_tuv);
int crt_trace_any(crt_ctx* ctx, crt_geometry g, size_t n, const float* d_org, const float* d_dir, float tmin,
                  float tmax, int32_t* d_out_hit);
/* same queries by exhaustive search over the triangle array with the reference's own test
 * (common/core.hpp:91-136): the GPU-side check that the BVH only culls */
int crt_trace_closest_brute(crt_ctx* ctx, const crt_triangle* d_triangles, size_t n_tris, size_t n,
                            const float* d_org, const float* d_dir, float tmin, float tmax, int32_t* d_out_prim,
                            float* d_out_tuv);

/* ---- kernels: one export per reference KERNEL, parameter lists verbatim (same order, same by-value
 * structs); grid/block are implied (the reference always launches ceil(W*H/256) x 256).
 * Reservoir / Visibility buffers are the reference's AoS layouts ("drop-in mode"). */
/* examples/10_restir_di/10_restir_di.cu:9-34.  When `triangles` is the array `geom` was built over, every pixel's walk
 * is first seeded with the triangle its record in `visibility_buffer` names on entry (last frame's answer for a host
 * that traces into the same buffer every frame; any content is allowed and none changes the result, which is the
 * exhaustive loop's closest hit bit for bit).  That array must then stay alive as long as `geom` is in use, as for
 * crt_refit_geometry.  CRT_RAYCAST_HINT=0 in the environment turns the seeding off. */
int crt_raycast(crt_ctx* ctx, int width, int height, crt_geometry geom, crt_buffer triangles, crt_raygen raygen,
                crt_buffer visibility_buffer);
/* 10_restir_di.cu:36-135 */
int crt_generate_candidate(crt_ctx* ctx, int width, int height, int frame, crt_geometry geom, crt_buffer triangles,
                           crt_buffer visibility_buffer, crt_float3 eye, crt_buffer lights, crt_options options,
                           crt_buffer reservoirs);
/* 10_restir_di.cu:137-237 */
int crt_temporal_resampling(crt_ctx* ctx, int width, int height, int frame, crt_geometry geom, crt_buffer triangles,
                            crt_buffer visibility_buffer, crt_float3 eye, crt_options options,
                            crt_buffer previous_reservoirs, crt_buffer reservoirs);
/* Extension (SURVEY.md section 8 f2; the reference has no counterpart: 10_restir_di.cu:174-180 reads the same pixel_idx and
 * 10_restir_di.cpp:257-267 only clears the accumulation when the camera moves).  temporal_resampling with the previous
 * reservoir read at the pixel the current surface point had in the previous frame's camera `previous_raygen`
 * (RayGenerator::shoot inverted, nearest sample point; no history behind that camera or outside its image); everything
 * else — M cap, rejection heuristics, merge, random stream — is the reference kernel's.  With an unmoved camera the
 * result equals crt_temporal_resampling bit for bit.  Specification: oracle/port/oracle_port.cpp: reproject_pixel.
 * This is the launch-list form (`previous_reservoirs` and `reservoirs` must be different buffers); with row slabs the
 * rows of `previous_reservoirs` a slab reads are no longer bounded by the spatial halo (the host must provide all rows
 * the camera motion can reach).  crt_launch name: "temporal_resampling_reprojected" (previous_raygen is the 9th param). */
int crt_temporal_resampling_reprojected(crt_ctx* ctx, int width, int height, int frame, crt_geometry geom, crt_buffer triangles,
                                        crt_buffer visibility_buffer, crt_float3 eye, crt_options options,
                                        crt_raygen previous_raygen, crt_buffer previous_reservoirs, crt_buffer reservoirs);
/* The same look-up inside the fused frame (crt_restir_frame_begin / crt_restir_di_frame): with a previous camera set,
 * the frame's candidate + temporal kernel reads the history at the reprojected pixel — from a snapshot of `temporal`
 * the library takes at the start of the frame (72 bytes per pixel of its own; the fused merge writes `temporal` in
 * place) — and with options that take the per-kernel path the call above is used.  NULL: no reprojection (the
 * reference's behaviour, the default).  A context that renders a row range (crt_set_row_range) must hold every row of
 * `temporal` the look-ups can reach: the host gathers the other contexts' rows before crt_restir_frame_begin
 * (python/slabs.py: SlabRenderer(reproject=True).gather_history does, over NCCL); the direct-store slab links mirror
 * the 87 halo rows only and the call refuses them.  With the previous camera equal to the current one the frame equals
 * the plain fused frame bit for bit. */
int crt_restir_set_previous_camera(crt_ctx* ctx, const crt_raygen* previous_raygen);
/* Reprojection that also receives the previous frame's surfaces (extension; DESIGN.md section 15, "Reprojection"): what
 * CRT_REUSE_UNBIASED needs with a moving camera.  crt_temporal_resampling_reprojected with one more input,
 * `previous_visibility_buffer`: last frame's Visibility buffer, which the host keeps for one more frame instead of tracing
 * over it (two Visibility buffers, alternated).  It is read at the history pixel h only.  Under CRT_REUSE_UNBIASED the
 * history's surface is S_h = make_surface_info of that record with the previous eye (previous_raygen.m_origin), its
 * confidence c_h = trunc(min(M_h, 20 * ris_sample_count) * rejection_heuristics(S_q, S_h)) with this frame's eye (0 when
 * h has no history, is sky, or M_h = 0), the history merges with weight p_hat_q(y_h) * ucw_h * c_h, M accumulates c_h, and
 *   Z = c_own [p_hat_q(y) > 0] + c_h [p_hat_h(y) > 0],   ucw = p_hat_q(y) > 0 && Z > 0 ? w_sum / (Z p_hat_q(y)) : 0
 * with p_hat_h the target function at S_h (a shadow ray from S_h under use_shadowed_target_function, traced only when
 * the unshadowed value is positive).  With an unmoved camera and this frame's Visibility as the previous one it equals
 * crt_temporal_resampling under CRT_REUSE_UNBIASED bit for bit.  Under CRT_REUSE_REFERENCE the previous Visibility is
 * not read and the result equals crt_temporal_resampling_reprojected bit for bit.  Unbiased for static geometry.
 * CRT_EINVAL: a buffer smaller than width * height, `previous_visibility_buffer` equal to `visibility_buffer`, or
 * `previous_reservoirs` equal to `reservoirs`.  Row ranges: the host provides every row of `previous_reservoirs` and
 * `previous_visibility_buffer` the look-ups can reach.  crt_launch name: "temporal_resampling_reprojected_surfaces"
 * (previous_visibility_buffer is the 10th param). */
int crt_temporal_resampling_reprojected_surfaces(crt_ctx* ctx, int width, int height, int frame, crt_geometry geom,
                                                 crt_buffer triangles, crt_buffer visibility_buffer, crt_float3 eye,
                                                 crt_options options, crt_raygen previous_raygen,
                                                 crt_buffer previous_visibility_buffer, crt_buffer previous_reservoirs,
                                                 crt_buffer reservoirs);
/* The same inside the fused frame: crt_restir_set_previous_camera plus the previous frame's Visibility buffer, which the
 * context stores (not copies) until it is cleared: the host keeps it unchanged until the next crt_restir_frame_begin has
 * run.  NULL previous_raygen clears both; crt_restir_set_previous_camera clears the stored Visibility.  Under
 * CRT_REUSE_UNBIASED crt_restir_frame_begin accepts a previous camera only when it was set here.  The frame checks
 * (CRT_EINVAL) that the buffer holds width * height records and is not buffers->visibility, which its raycast
 * overwrites; options that take the per-kernel path use crt_temporal_resampling_reprojected_surfaces.  On a row range the
 * fused frame with unbiased weights needs crt_restir_set_halo_surfaces, and the host provides every row of `temporal` and
 * of the previous Visibility the look-ups can reach (python/slabs.py: SlabRenderer(reproject="surfaces")). */
int crt_restir_set_previous_frame(crt_ctx* ctx, const crt_raygen* previous_raygen, crt_buffer previous_visibility);
/* Reprojection that follows moving geometry (extension; DESIGN.md section 17): crt_temporal_resampling_reprojected_surfaces
 * with one more input, `previous_triangles`: the triangle array of the previous frame, the same count and order as
 * `triangles` (a host that writes vertices and calls crt_refit_geometry keeps the outgoing array for one frame).  For a
 * pixel with Visibility (prim, u, v) the look-up projects the point's previous position into the previous camera: the
 * surface point itself when the 36 vertex bytes of `prim` are equal in both arrays, otherwise the same barycentrics on
 * the previous vertices.  Under CRT_REUSE_UNBIASED the history's surface S_h is built from the previous Visibility at h
 * on the previous array's triangle when that triangle's vertex bytes differ, on `triangles` otherwise; the merge is
 * crt_temporal_resampling_reprojected_surfaces'.  With `previous_triangles` byte-equal to `triangles` the result equals
 * crt_temporal_resampling_reprojected_surfaces (CRT_REUSE_UNBIASED) or crt_temporal_resampling_reprojected
 * (CRT_REUSE_REFERENCE) bit for bit.  Under CRT_REUSE_REFERENCE `previous_visibility_buffer` is not read and may be empty.
 * The merged history is then the one built at the same material point; unbiasedness is as for
 * crt_temporal_resampling_reprojected_surfaces with static emitters and the unshadowed target function (DESIGN.md
 * section 17, "Scope" and "What the test can see").
 * CRT_EINVAL: the refusals of crt_temporal_resampling_reprojected_surfaces, `previous_triangles` of another size than
 * `triangles` or null with a nonzero size, and CRT_REUSE_UNBIASED without a previous Visibility buffer.  crt_launch name:
 * "temporal_resampling_reprojected_motion" (previous_triangles is the 10th param, previous_visibility_buffer the 11th). */
int crt_temporal_resampling_reprojected_motion(crt_ctx* ctx, int width, int height, int frame, crt_geometry geom,
                                               crt_buffer triangles, crt_buffer visibility_buffer, crt_float3 eye,
                                               crt_options options, crt_raygen previous_raygen, crt_buffer previous_triangles,
                                               crt_buffer previous_visibility_buffer, crt_buffer previous_reservoirs,
                                               crt_buffer reservoirs);
/* The same inside the fused frame: the previous frame's triangle array, which the context stores (not copies) until it is
 * cleared; the host keeps it unchanged until the next crt_restir_frame_begin has run.  NULL data clears it, and so does a
 * NULL previous_raygen passed to crt_restir_set_previous_camera or crt_restir_set_previous_frame.  It applies while a
 * previous camera is set: crt_restir_frame_begin then checks (CRT_EINVAL) that it holds as many triangles as `triangles`,
 * and options that take the per-kernel path use crt_temporal_resampling_reprojected_motion.  CRT_EINVAL: null data with a
 * nonzero size. */
int crt_restir_set_previous_triangles(crt_ctx* ctx, crt_buffer previous_triangles);
/* Halo surfaces (extension; DESIGN.md section 15, "Halo surfaces"; off by default): what the fused frame with
 * CRT_REUSE_UNBIASED needs on a row range narrower than the image or with slab links.  Its spatial passes read every
 * visited neighbour's primary-hit surface from the context's G-buffer, which the candidate kernel writes for the context's
 * own rows only.  With this on, under CRT_REUSE_UNBIASED and fused options, crt_restir_frame_begin also produces the records
 * of rows [y0 - h, y0) and [y1, y1 + h), clipped to the image, h = the rows a pass of spatial_resampling_radius can reach
 * (87 at radius 30): primary rays into a Visibility buffer of the context's own (the host's buffers are written in the
 * context's own rows only, as always), then the surface of every diffuse pixel with this frame's eye — bit for bit what
 * the context that owns the row stores.  crt_restir_spatial_pass refuses (CRT_EINVAL) a radius that reaches further than
 * the frame's begin covered.  The reservoirs of halo rows still come from the host's exchange or the slab links, whose own
 * constraints stay (radius <= 30, spatial_resampling_passes != 1, slabs at least 87 rows tall).  Under
 * CRT_REUSE_REFERENCE, on the whole image, or without spatial passes nothing is launched and every result is unchanged. */
int crt_restir_set_halo_surfaces(crt_ctx* ctx, int enable);
/* 10_restir_di.cu:239-254 — note the reference's parameter names are swapped: the first buffer is the source */
int crt_save_temporal_reservoir(crt_ctx* ctx, int width, int height, crt_buffer src, crt_buffer dst);
/* 10_restir_di.cu:256-388 */
int crt_spatial_resampling(crt_ctx* ctx, int width, int height, int frame, int pass, crt_geometry geom,
                           crt_buffer triangles, crt_buffer visibility_buffer, crt_float3 eye, crt_options options,
                           crt_buffer previous_reservoirs, crt_buffer reservoirs);
/* 10_restir_di.cu:390-459 */
int crt_resolve(crt_ctx* ctx, crt_buffer accumulation, int width, int height, crt_geometry geom,
                crt_buffer triangles, crt_buffer visibility_buffer, crt_float3 eye, crt_options options,
                crt_buffer reservoirs);
/* common/kernels/common.cu:4-17 and :30-74 */
int crt_clear(crt_ctx* ctx, crt_buffer buffer, int width, int height);
int crt_tone_mapping(crt_ctx* ctx, crt_buffer pixels, crt_buffer accumulation, int width, int height);
/* examples/07_pt/07_pt.cu:11-15, 08_nee/08_nee.cu:11-15, 09_ris/09_ris.cu:11-15 */
int crt_path_trace_07(crt_ctx* ctx, int width, int height, int frame, crt_geometry geom, crt_buffer triangles,
                      crt_raygen raygen, crt_options options, crt_buffer accumulation);
int crt_path_trace_08(crt_ctx* ctx, int width, int height, int frame, crt_geometry geom, crt_buffer triangles,
                      crt_buffer lights, crt_raygen raygen, crt_options options, crt_buffer accumulation);
int crt_path_trace_09(crt_ctx* ctx, int width, int height, int frame, crt_geometry geom, crt_buffer triangles,
                      crt_buffer lights, crt_raygen raygen, crt_options options, crt_buffer accumulation);
/* examples/06_ao_hiprt/06_ao_hiprt.cu:35-37; n_rays replaces the hard-coded N_Rays = 64 (:71) */
int crt_ao_06(crt_ctx* ctx, crt_buffer pixels, crt_raygen raygen, int width, int height, crt_geometry geom,
              crt_buffer triangles, int n_rays);

/* ---- fused frame ("fast mode").  One call replaces the launch list of a frame
 * (examples/10_restir_di/10_restir_di.cpp:270-372: raycast ... tone_mapping) with identical results in
 * `accumulation`, `pixels` and `visibility`.  The three TypedBuffer<Reservoir> allocations (W*H*76 bytes each, as
 * the reference allocates them, :112-122) are used as OPAQUE storage: inside, reservoirs are sector-planar
 *   plane 0 at byte offset 0 and plane 1 at 32*W*H, 32 bytes per pixel; plane 2 at 64*W*H, 8 bytes per pixel
 *   (field order and flag bits: csrc/restir_fast.cuh), pixel order = the reference's pixel_idx (bottom-up rows),
 * candidate generation and temporal resampling are one kernel that rewrites `temporal` in place (no
 * save_temporal_reservoir), spatial pass 0 reads `temporal` and writes reservoir1, later passes ping-pong
 * reservoir1 <-> reservoir0, and tone mapping is part of resolve.  crt_reservoir_export_aos converts a buffer to
 * the reference's AoS for inspection.  With use_shadowed_target_function (or option values that would let M pass
 * 2^29) the same calls run the per-kernel path on AoS buffers instead (crt_restir_is_fused tells which); do not mix
 * the two on one set of buffers.  resolve does not re-trace a shadow ray whose answer the history already holds
 * (same origin, same target, same geometry: csrc/restir_fast.cuh kTracedBit); CRT_RESOLVE_REUSE=0 in the
 * environment of crt_init makes it trace every ray like the reference.  Images are bit-identical either way. */
typedef struct
{
    crt_buffer pixels;        /* TypedBuffer<uint8_t>   4*W*H   (10_restir_di.cpp:96-97)  */
    crt_buffer accumulation;  /* TypedBuffer<float4>    W*H     (:102-103) */
    crt_buffer visibility;    /* TypedBuffer<Visibility> W*H    (:108-109) */
    crt_buffer reservoir0;    /* TypedBuffer<Reservoir> W*H     (:113-114) */
    crt_buffer reservoir1;    /*                                (:117-118) */
    crt_buffer temporal;      /* zero it once before frame 1    (:121-122) */
} crt_restir_buffers;
int crt_restir_di_frame(crt_ctx* ctx, int width, int height, int frame, crt_geometry geom, crt_buffer triangles,
                        crt_raygen raygen, crt_float3 eye, crt_buffer lights, crt_options options,
                        const crt_restir_buffers* buffers);
/* the same frame in three stages, for hosts that exchange halo rows between them (multi-GPU row slabs):
 * begin = raycast + candidates + temporal; one call per spatial pass; end = resolve + tone mapping */
int crt_restir_frame_begin(crt_ctx* ctx, int width, int height, int frame, crt_geometry geom, crt_buffer triangles,
                           crt_raygen raygen, crt_float3 eye, crt_buffer lights, crt_options options,
                           const crt_restir_buffers* buffers);
int crt_restir_spatial_pass(crt_ctx* ctx, int width, int height, int frame, int pass, crt_geometry geom,
                            crt_buffer triangles, crt_float3 eye, crt_options options,
                            const crt_restir_buffers* buffers);
int crt_restir_frame_end(crt_ctx* ctx, int width, int height, crt_geometry geom, crt_buffer triangles, crt_float3 eye,
                         crt_options options, const crt_restir_buffers* buffers);
/* which of the three buffers holds the reservoirs resolve reads (the reference's buf_output, :324-336) */
int crt_restir_output_buffer(crt_options options, const crt_restir_buffers* buffers, crt_buffer* out);
int crt_restir_is_fused(crt_options options);
/* device pointer to the W*H-byte pixel-class plane of the last fused frame (1 = diffuse surface, 0 = sky or
 * emissive): the only per-frame data besides reservoir rows a multi-GPU host has to exchange */
int crt_restir_class_plane(crt_ctx* ctx, void** out);
int crt_reservoir_export_aos(crt_ctx* ctx, int width, int height, crt_buffer soa_storage, crt_buffer aos_out);
int crt_reservoir_import_aos(crt_ctx* ctx, int width, int height, crt_buffer aos_in, crt_buffer soa_storage);

/* ---- multi-GPU row slabs: halo rows by direct peer stores (new; the reference is single-GPU).
 * One process per GPU.  Each rank allocates its three reservoir buffers with crt_malloc, calls
 * crt_restir_reserve, exports both with crt_ipc_export (cudaIpc handles, 64 bytes, to be passed to the neighbour
 * ranks by any host channel), opens its neighbours' handles and registers the peer pointers with
 * crt_slab_set_links.  crt_slab_exchange then replaces the host-side halo exchange between the stages of the fused
 * frame: it stores this rank's 87 boundary rows of the chosen buffer into the neighbours' buffers over NVLink,
 * signals them, and waits for their rows (csrc/slab_p2p.cu).  Constraints, all checked (CRT_EINVAL): slabs at least
 * 87 rows tall, image width a multiple of 16, spatial_resampling_radius <= 30 (the mirrored band is 87 rows: the
 * reach of radius 30), options that run the fused bodies (crt_restir_is_fused), and 0 or >= 2 spatial passes — the
 * one signal/wait per pass is the only ordering between neighbours, and with a single pass a neighbour's next frame
 * could overwrite halo rows this slab is still reading.  Anything else: exchange the rows on the host side
 * (python/slabs.py does it with NCCL).  Unmap the neighbours' buffers (crt_slab_set_links(NULL), crt_ipc_close) before
 * any rank frees the buffers it exported. */
int crt_ipc_export(crt_ctx* ctx, void* device_ptr, unsigned char handle_out[64]);
int crt_ipc_open(crt_ctx* ctx, const unsigned char handle[64], void** peer_ptr_out);
int crt_ipc_close(crt_ctx* ctx, void* peer_ptr);
/* allocates the fused frame's per-pixel scratch for a W x H image now (instead of at the first frame) and returns
 * the base of that allocation; the pixel-class plane is the W*H bytes at offset 24*W*H */
int crt_restir_reserve(crt_ctx* ctx, int width, int height, void** scratch_base_out);
typedef struct
{
    /* peer pointers into the slab above (smaller yi) / below: [0] temporal, [1] reservoir0, [2] reservoir1 storage,
     * [3] pixel-class plane; all NULL = no neighbour on that side */
    void* up[4];
    void* down[4];
    void* up_flag;   /* 8-byte slot this rank raises in the upper neighbour's flag buffer (its slot 1) */
    void* down_flag; /* ... in the lower neighbour's flag buffer (its slot 0) */
    void* my_flags;  /* this rank's own flag buffer: 32 zeroed bytes — slot 0 (raised by `up`), slot 1 (raised by `down`),
                      * the 8-byte time-out mark crt_slab_status reads, 8 bytes reserved */
} crt_slab_links;
int crt_slab_set_links(crt_ctx* ctx, const crt_slab_links* links);
/* Call between the stages of the fused frame, before the spatial pass that reads buffer `which` (0 temporal,
 * 1 reservoir0, 2 reservoir1).  While links are set, crt_restir_frame_begin / crt_restir_spatial_pass already
 * mirror their boundary rows into the neighbours' buffers, so push_rows = 0 only signals the neighbours and waits
 * for theirs; push_rows = 1 first copies the 87 boundary rows of the buffer with a dedicated kernel, 2 also the
 * pixel-class rows (for buffers filled by other means). */
/* 0, or the exchange count at which a wait for a neighbour gave up after 4 s (the frame is then invalid); waits for the
 * stream.  The flag buffer registered with crt_slab_set_links is 32 bytes: two slots and this mark. */
int crt_slab_status(crt_ctx* ctx, unsigned long long* timed_out_stage);
int crt_slab_exchange(crt_ctx* ctx, int width, int height, int which, int push_rows,
                      const crt_restir_buffers* buffers);

/* Shader::launch call shape (common/shader.hpp:179-199): kernel by name, params as the void*[] that
 * ShaderArgument builds (pointers to by-value arguments, in order), grid/block accepted and ignored.
 * Names: raycast, generate_candidate, temporal_resampling, save_temporal_reservoir, spatial_resampling,
 * resolve, clear, tone_mapping (example 10); path_trace_07/08/09; ao_06 (its 7th param is int n_rays). */
int crt_launch(crt_ctx* ctx, const char* name, void** params, unsigned gx, unsigned gy, unsigned gz, unsigned bx,
               unsigned by, unsigned bz);

#ifdef __cplusplus
}
#endif
#endif /* CEDECRT_H */
