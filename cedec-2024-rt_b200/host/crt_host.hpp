// crt_host.hpp — C++ host layer over the C ABI (include/cedecrt.h) with the reference's host-side names, so a
// main() written against common/typedbuffer.hpp + common/shader.hpp + common/loader.hpp of the reference keeps
// its shape:
//
//   reference                                           here
//   oroInitialize/oroCtxCreate/oroStreamCreate          crt::Device dev(0);                      (10_restir_di.cpp:30-53)
//   TypedBuffer<T> b(TYPED_BUFFER_DEVICE); b.allocate   TypedBuffer<T> b(dev); b.allocate(n);    (typedbuffer.hpp:29-77)
//   Shader shader(file, label, options, UseHiprt(..))   Shader shader(dev);   (nothing to compile at run time)
//   shader.launch(name, ShaderArgument()..., grid...)   same call                                (shader.hpp:179-199)
//   buildHiprtGeometry(hContext, triangles)             buildGeometry(dev, triangle_buffer)      (loader.hpp:68-112)
//   OroStopwatch sw(stream); sw.start/stop/getMs        Stopwatch sw(dev); same calls            (OrochiUtils.h:179-209)
//
// Errors: every failing C-ABI call throws crt::Error carrying crt_last_error() — the reference ignores Orochi
// return codes or raises SIGTRAP through SH_ASSERT (shader.hpp:10-16).  There is no CPU path: constructing a
// Device without a CUDA device throws.
#pragma once
#include <cstdint>
#include <cstdio>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/cedecrt.h"

namespace crt
{
struct Error : std::runtime_error
{
    int code;
    Error(int c, const std::string& what) : std::runtime_error(what), code(c) {}
};
inline void check(int rc, const char* call)
{
    if (rc != CRT_OK) throw Error(rc, std::string(call) + " failed (" + std::to_string(rc) + "): " + crt_last_error());
}
#define CRT_CHECKED(call) ::crt::check((call), #call)

// one GPU: device + stream (crt_ctx)
class Device
{
   public:
    explicit Device(int index = 0) { CRT_CHECKED(crt_init(index, &m_ctx)); }
    ~Device() { crt_shutdown(m_ctx); }
    Device(const Device&) = delete;
    Device& operator=(const Device&) = delete;
    crt_ctx* ctx() const { return m_ctx; }
    const char* name() const { return crt_device_name(m_ctx); }
    void synchronize() const { CRT_CHECKED(crt_sync(m_ctx)); }
    void setRowRange(int y0, int y1) const { CRT_CHECKED(crt_set_row_range(m_ctx, y0, y1)); }
    // CRT_LIGHTS_UNIFORM (the reference) or CRT_LIGHTS_POWER; log2_slots = 0: the default slot count
    void setLightSampling(int mode, int log2_slots = 0) const { CRT_CHECKED(crt_set_light_sampling(m_ctx, mode, log2_slots)); }
    // presampled light tiles for the ReSTIR DI candidates: 2^log2_tiles tiles of 2^log2_tile_size records; (0, 0): off
    void setLightTiles(int log2_tiles, int log2_tile_size) const { CRT_CHECKED(crt_set_light_tiles(m_ctx, log2_tiles, log2_tile_size)); }
    // CRT_REUSE_REFERENCE (the reference) or CRT_REUSE_UNBIASED (1/Z weights in every temporal and spatial merge)
    void setReuseWeights(int mode) const { CRT_CHECKED(crt_set_reuse_weights(m_ctx, mode)); }
    // temporal reprojection in the fused frame with the previous frame's Visibility buffer (what CRT_REUSE_UNBIASED needs
    // with a moving camera); the host keeps that buffer until the next frame has begun.  nullptr clears both.
    void setPreviousFrame(const crt_raygen* previous_raygen, crt_buffer previous_visibility) const
    {
        CRT_CHECKED(crt_restir_set_previous_frame(m_ctx, previous_raygen, previous_visibility));
    }
    // the fused frame with CRT_REUSE_UNBIASED on a row range or with slab links: frame begin also produces the G-buffer
    // records of the halo rows its spatial passes read; nothing changes under the reference's weights
    void setHaloSurfaces(bool enable) const { CRT_CHECKED(crt_restir_set_halo_surfaces(m_ctx, enable ? 1 : 0)); }
    // moving geometry in the fused frame's reprojection: the previous frame's triangle array (same count and order), kept
    // by the host until the next frame has begun; an empty buffer clears it
    void setPreviousTriangles(crt_buffer previous_triangles) const
    {
        CRT_CHECKED(crt_restir_set_previous_triangles(m_ctx, previous_triangles));
    }
    // the launch list's reprojected temporal resampling with the previous frame's Visibility buffer
    void temporalResamplingReprojectedSurfaces(int width, int height, int frame, crt_geometry geom, crt_buffer triangles,
                                               crt_buffer visibility, crt_float3 eye, crt_options options,
                                               crt_raygen previous_raygen, crt_buffer previous_visibility,
                                               crt_buffer previous_reservoirs, crt_buffer reservoirs) const
    {
        CRT_CHECKED(crt_temporal_resampling_reprojected_surfaces(m_ctx, width, height, frame, geom, triangles, visibility, eye,
                                                                 options, previous_raygen, previous_visibility,
                                                                 previous_reservoirs, reservoirs));
    }

   private:
    crt_ctx* m_ctx = nullptr;
};
}  // namespace crt

// Device-resident TypedBuffer<T>.  The first 16 bytes are the reference's {T* m_data; size_t m_size:63,
// m_isDevice:1} (typedbuffer.hpp:14-20): ShaderArgument::ptr(&buffer) hands exactly those bytes to the kernel.
template <class T>
struct TypedBuffer
{
    T* m_data = nullptr;
    size_t m_size : 63;
    size_t m_isDevice : 1;
    const crt::Device* m_dev;

    explicit TypedBuffer(const crt::Device& dev) : m_size(0), m_isDevice(1), m_dev(&dev) {}
    TypedBuffer(const TypedBuffer&) = delete;
    void operator=(const TypedBuffer&) = delete;
    ~TypedBuffer()
    {
        if (m_data) crt_free(m_dev->ctx(), m_data);
    }
    void allocate(size_t n)  // uninitialised, like oroMalloc
    {
        if (m_data) CRT_CHECKED(crt_free(m_dev->ctx(), m_data));
        m_data = nullptr;
        void* p = nullptr;
        CRT_CHECKED(crt_malloc(m_dev->ctx(), n * sizeof(T), &p));
        m_data = (T*)p;
        m_size = n;
    }
    void zero() { CRT_CHECKED(crt_memset(m_dev->ctx(), m_data, 0, bytes())); }
    void upload(const T* src, size_t n)  // oroMemcpyHtoD (10_restir_di.cpp:211,216)
    {
        if (n > m_size) throw crt::Error(CRT_EINVAL, "TypedBuffer::upload: source larger than the buffer");
        CRT_CHECKED(crt_memcpy_h2d(m_dev->ctx(), m_data, src, n * sizeof(T)));
    }
    std::vector<T> toHost() const
    {
        std::vector<T> out(m_size);
        CRT_CHECKED(crt_memcpy_d2h(m_dev->ctx(), out.data(), m_data, bytes()));
        return out;
    }
    size_t size() const { return m_size; }
    size_t bytes() const { return m_size * sizeof(T); }
    T* data() { return m_data; }
    const T* data() const { return m_data; }
};
static_assert(sizeof(size_t) == 8, "64-bit host expected");

// ShaderArgument (shader.hpp:42-87): value() copies a POD, ptr() passes the pointee's bytes by value
struct ShaderArgument
{
    template <class T>
    ShaderArgument& value(const T& v)
    {
        auto* holder = new Holder<T>(v);
        m_owned.emplace_back(holder);
        m_params.push_back(&holder->v);
        return *this;
    }
    template <class T>
    ShaderArgument& ptr(T* p)
    {
        m_params.push_back((void*)p);
        return *this;
    }
    void** kernelParams() const { return const_cast<void**>(m_params.data()); }

   private:
    struct HolderBase
    {
        virtual ~HolderBase() {}
    };
    template <class T>
    struct Holder : HolderBase
    {
        explicit Holder(const T& x) : v(x) {}
        T v;
    };
    std::vector<std::unique_ptr<HolderBase>> m_owned;
    std::vector<void*> m_params;
};

// Shader::launch (shader.hpp:179-199).  Kernels are precompiled for sm_100a inside libcedecrt.so, so the
// constructor has nothing to compile; grid/block arguments are accepted and ignored.
class Shader
{
   public:
    explicit Shader(const crt::Device& dev) : m_dev(&dev) {}
    void launch(const char* name, const ShaderArgument& args, unsigned gx, unsigned gy, unsigned gz, unsigned bx,
                unsigned by, unsigned bz, void* /*stream*/ = nullptr) const
    {
        crt::check(crt_launch(m_dev->ctx(), name, args.kernelParams(), gx, gy, gz, bx, by, bz), name);
    }

   private:
    const crt::Device* m_dev;
};

// buildHiprtGeometry (loader.hpp:68-112): BVH over the device-resident triangle array, synchronous
inline crt_geometry buildGeometry(const crt::Device& dev, const TypedBuffer<crt_triangle>& triangles)
{
    crt_geometry g = nullptr;
    CRT_CHECKED(crt_build_geometry(dev.ctx(), triangles.data(), triangles.size(), &g));
    return g;
}

// hiprtBuildOperationUpdate (hiprt_types.h:131-135): the host moved vertices in `triangles` (same count and order)
inline void refitGeometry(const crt::Device& dev, crt_geometry geom) { CRT_CHECKED(crt_refit_geometry(dev.ctx(), geom)); }

// OroStopwatch (OrochiUtils.h:179-209)
class Stopwatch
{
   public:
    explicit Stopwatch(const crt::Device& dev) : m_dev(&dev) {}
    void start() { CRT_CHECKED(crt_timer_start(m_dev->ctx())); }
    void stop() { CRT_CHECKED(crt_timer_stop_ms(m_dev->ctx(), &m_ms)); }
    float getMs() const { return m_ms; }

   private:
    const crt::Device* m_dev;
    float m_ms = 0.0f;
};

inline int ceiling_div(int a, int b) { return (a + b - 1) / b; }  // common/math.hpp:174-181
