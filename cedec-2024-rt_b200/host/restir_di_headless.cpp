// restir_di_headless.cpp — the application loop of examples/10_restir_di/10_restir_di.cpp (229-413) without a
// window: same buffers, same launch list through Shader::launch, same per-frame "kernel: x ms" timing
// (OroStopwatch around the launch list), RGBA8 copied back every frame; the last frame is written as a PPM.
//
//   restir_di_headless --scene assets/blocks_restir.tri[.xz] [--tile NX NZ DX DZ] [--size W H] [--frames N]
//                      [--eye x y z] [--lookat x y z] [--no-temporal] [--no-spatial] [--no-accumulate]
//                      [--out image.ppm] [--dump-accum file.f32] [--fused] [--lights uniform|power]
//                      [--reuse reference|unbiased] [--light-tiles LOG2_T LOG2_S]
//
// --fused issues one crt_restir_di_frame call per frame instead of the launch list (same image, see cedecrt.h).
//
// --scene takes the raw bytes of a std::vector<Triangle> as the reference loader produces it (assets/*.tri;
// .xz is piped through `xz -dc`) or, with a name ending in .obj, a Wavefront OBJ read by obj_scene.hpp.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "crt_host.hpp"
#include "obj_scene.hpp"

static std::vector<crt_triangle> load_tri_cache(const std::string& path)
{
    const bool xz = path.size() > 3 && path.compare(path.size() - 3, 3, ".xz") == 0;
    FILE* f = xz ? popen(("xz -dc '" + path + "'").c_str(), "r") : fopen(path.c_str(), "rb");
    if (!f) throw crt::Error(CRT_EINVAL, "cannot open scene " + path);
    std::vector<crt_triangle> tris;
    std::vector<char> chunk(60 * 65536);
    std::vector<char> all;
    size_t got;
    while ((got = fread(chunk.data(), 1, chunk.size(), f)) > 0) all.insert(all.end(), chunk.begin(), chunk.begin() + got);
    xz ? pclose(f) : fclose(f);
    if (all.empty() || all.size() % sizeof(crt_triangle)) throw crt::Error(CRT_EINVAL, "scene " + path + ": not a Triangle[] file");
    tris.resize(all.size() / sizeof(crt_triangle));
    memcpy(tris.data(), all.data(), all.size());
    return tris;
}

int main(int argc, char** argv)
{
    std::string scene, out_ppm, dump_accum;
    bool fused = false;
    int light_mode = CRT_LIGHTS_UNIFORM;  // --lights power: select lights in proportion to their power (cedecrt.h)
    int reuse_mode = CRT_REUSE_REFERENCE;  // --reuse unbiased: 1/Z weights in the temporal and spatial merges (cedecrt.h)
    int tiles_log2_t = 0, tiles_log2_s = 0;  // --light-tiles 7 10: the candidates draw from presampled light tiles (cedecrt.h)
    int width = 1920, height = 1080, frames = 4, tile_nx = 1, tile_nz = 1;
    float tile_dx = 130.0f, tile_dz = 82.0f;
    float eye[3] = {-0.579885f, 22.194597f, -6.567105f}, center[3] = {5.224952f, 20.847435f, 1.431192f};  // :188-189
    crt_options options;
    memset(&options, 0, sizeof options);  // common/options.hpp:4-23 defaults, then the ReSTIR toggles on
    options.max_depth = 6;
    options.ris_sample_count = 32;
    options.rejection_heuristics_threshold = 0.2f;
    options.spatial_resampling_sample_count = 5;
    options.spatial_resampling_radius = 30.0f;
    options.spatial_resampling_passes = 3;
    options.use_visibility_reuse = 1;
    options.accumulate = 1;
    options.use_temporal_resampling = 1;
    options.use_spatial_resampling = 1;
    for (int i = 1; i < argc; i++)
    {
        const std::string a = argv[i];
        auto need = [&](int n) {
            if (i + n >= argc)
            {
                fprintf(stderr, "%s: missing value\n", a.c_str());
                exit(2);
            }
        };
        if (a == "--scene") { need(1); scene = argv[++i]; }
        else if (a == "--size") { need(2); width = atoi(argv[++i]); height = atoi(argv[++i]); }
        else if (a == "--frames") { need(1); frames = atoi(argv[++i]); }
        else if (a == "--tile") { need(4); tile_nx = atoi(argv[++i]); tile_nz = atoi(argv[++i]); tile_dx = (float)atof(argv[++i]); tile_dz = (float)atof(argv[++i]); }
        else if (a == "--eye") { need(3); for (int k = 0; k < 3; k++) eye[k] = (float)atof(argv[++i]); }
        else if (a == "--lookat") { need(3); for (int k = 0; k < 3; k++) center[k] = (float)atof(argv[++i]); }
        else if (a == "--no-temporal") options.use_temporal_resampling = 0;
        else if (a == "--no-spatial") options.use_spatial_resampling = 0;
        else if (a == "--no-accumulate") options.accumulate = 0;
        else if (a == "--fused") fused = true;
        else if (a == "--lights")
        {
            need(1);
            const std::string m = argv[++i];
            if (m != "uniform" && m != "power")
            {
                fprintf(stderr, "--lights takes uniform or power\n");
                return 2;
            }
            light_mode = m == "power" ? CRT_LIGHTS_POWER : CRT_LIGHTS_UNIFORM;
        }
        else if (a == "--reuse")
        {
            need(1);
            const std::string m = argv[++i];
            if (m != "reference" && m != "unbiased")
            {
                fprintf(stderr, "--reuse takes reference or unbiased\n");
                return 2;
            }
            reuse_mode = m == "unbiased" ? CRT_REUSE_UNBIASED : CRT_REUSE_REFERENCE;
        }
        else if (a == "--light-tiles") { need(2); tiles_log2_t = atoi(argv[++i]); tiles_log2_s = atoi(argv[++i]); }
        else if (a == "--out") { need(1); out_ppm = argv[++i]; }
        else if (a == "--dump-accum") { need(1); dump_accum = argv[++i]; }
        else
        {
            fprintf(stderr, "unknown argument %s\n", a.c_str());
            return 2;
        }
    }
    if (scene.empty())
    {
        fprintf(stderr, "usage: %s --scene <file.tri[.xz]|file.obj> [--size W H] [--frames N] [--out image.ppm]\n", argv[0]);
        return 2;
    }
    try
    {
        crt::Device device(0);
        printf("Device: %s\n", device.name());
        device.setLightSampling(light_mode);
        device.setReuseWeights(reuse_mode);
        device.setLightTiles(tiles_log2_t, tiles_log2_s);
        Shader shader(device);

        std::vector<crt_triangle> triangles =
            scene.size() > 4 && scene.compare(scene.size() - 4, 4, ".obj") == 0 ? crt::loadTrianglesFromObj(scene) : load_tri_cache(scene);
        if (tile_nx * tile_nz > 1)  // BASELINE config 5: tile-major copies on an x,z grid
        {
            const size_t n = triangles.size();
            triangles.resize(n * tile_nx * tile_nz);
            for (int t = 1; t < tile_nx * tile_nz; t++)
                for (size_t k = 0; k < n; k++)
                {
                    crt_triangle tr = triangles[k];
                    for (auto& v : tr.vertices)
                    {
                        v.x += (float)(t % tile_nx) * tile_dx;
                        v.z += (float)(t / tile_nx) * tile_dz;
                    }
                    triangles[(size_t)t * n + k] = tr;
                }
        }
        std::vector<uint32_t> light_indices;  // 10_restir_di.cpp:196-206
        for (size_t i = 0; i < triangles.size(); i++)
        {
            const crt_float3& e = triangles[i].emissive;
            if (e.x > 0.0f || e.y > 0.0f || e.z > 0.0f) light_indices.push_back((uint32_t)i);
        }
        printf("triangles: %zu\nlights: %zu\n", triangles.size(), light_indices.size());

        const size_t n = (size_t)width * height;
        TypedBuffer<uint8_t> pixel_buffer(device);
        pixel_buffer.allocate(4 * n);
        TypedBuffer<crt_float4> accumulation_buffer(device);
        accumulation_buffer.allocate(n);
        TypedBuffer<crt_visibility> visibility_buffer(device);
        visibility_buffer.allocate(n);
        TypedBuffer<crt_reservoir> reservoir_buffer0(device), reservoir_buffer1(device), temporal_reservoir_buffer(device);
        reservoir_buffer0.allocate(n);
        reservoir_buffer1.allocate(n);
        temporal_reservoir_buffer.allocate(n);
        temporal_reservoir_buffer.zero();  // the reference leaves it uninitialised (:121-122); zero = no history

        TypedBuffer<crt_triangle> triangle_buffer(device);
        triangle_buffer.allocate(triangles.size());
        triangle_buffer.upload(triangles.data(), triangles.size());
        TypedBuffer<uint32_t> light_buffer(device);
        light_buffer.allocate(light_indices.size());
        light_buffer.upload(light_indices.data(), light_indices.size());

        crt_geometry geom = buildGeometry(device, triangle_buffer);
        double stats[8];
        CRT_CHECKED(crt_geometry_stats(geom, stats));
        printf("bvh: %.0f wide nodes, depth %.0f, built in %.1f ms\n", stats[1], stats[2], stats[3]);

        const unsigned grid = (unsigned)ceiling_div(width * height, 256);
        shader.launch("clear", ShaderArgument().ptr(&accumulation_buffer).value(width).value(height), grid, 1, 1, 256, 1, 1);

        const float up[3] = {0.0f, 1.0f, 0.0f};
        const crt_float3 cameraOrig = {eye[0], eye[1], eye[2]};
        std::vector<uint8_t> host_pixels(4 * n);
        double total_ms = 0.0;
        for (int frame = 1; frame <= frames; frame++)
        {
            crt_raygen rayGen;
            crt_raygen_lookat(&rayGen, eye, center, up, 3.14159265358979323846f / 4.0f, width, height);
            Stopwatch sw(device);
            sw.start();
            if (fused)
            {
                auto view = [](auto& b) { return crt_buffer{b.data(), b.size() | (1ull << 63)}; };
                const crt_restir_buffers bufs = {view(pixel_buffer), view(accumulation_buffer), view(visibility_buffer),
                                                 view(reservoir_buffer0), view(reservoir_buffer1), view(temporal_reservoir_buffer)};
                CRT_CHECKED(crt_restir_di_frame(device.ctx(), width, height, frame, geom, view(triangle_buffer), rayGen, cameraOrig,
                                                view(light_buffer), options, &bufs));
            }
            else
            {
            shader.launch("raycast",
                          ShaderArgument().value(width).value(height).value(geom).ptr(&triangle_buffer).ptr(&rayGen).ptr(&visibility_buffer),
                          grid, 1, 1, 256, 1, 1);
            shader.launch("generate_candidate",
                          ShaderArgument().value(width).value(height).value(frame).value(geom).ptr(&triangle_buffer)
                              .ptr(&visibility_buffer).value(cameraOrig).ptr(&light_buffer).value(options).ptr(&reservoir_buffer0),
                          grid, 1, 1, 256, 1, 1);
            shader.launch("temporal_resampling",
                          ShaderArgument().value(width).value(height).value(frame).value(geom).ptr(&triangle_buffer)
                              .ptr(&visibility_buffer).value(cameraOrig).value(options).ptr(&temporal_reservoir_buffer).ptr(&reservoir_buffer0),
                          grid, 1, 1, 256, 1, 1);
            shader.launch("save_temporal_reservoir",
                          ShaderArgument().value(width).value(height).ptr(&reservoir_buffer0).ptr(&temporal_reservoir_buffer),
                          grid, 1, 1, 256, 1, 1);
            TypedBuffer<crt_reservoir>* buf_input = &reservoir_buffer0;
            TypedBuffer<crt_reservoir>* buf_output = &reservoir_buffer1;
            for (int pass = 0; pass < options.spatial_resampling_passes; pass++)
            {
                if (pass != 0) std::swap(buf_input, buf_output);
                shader.launch("spatial_resampling",
                              ShaderArgument().value(width).value(height).value(frame).value(pass).value(geom).ptr(&triangle_buffer)
                                  .ptr(&visibility_buffer).value(cameraOrig).value(options).ptr(buf_input).ptr(buf_output),
                              grid, 1, 1, 256, 1, 1);
            }
            shader.launch("resolve",
                          ShaderArgument().ptr(&accumulation_buffer).value(width).value(height).value(geom).ptr(&triangle_buffer)
                              .ptr(&visibility_buffer).value(cameraOrig).value(options).ptr(buf_output),
                          grid, 1, 1, 256, 1, 1);
            shader.launch("tone_mapping", ShaderArgument().ptr(&pixel_buffer).ptr(&accumulation_buffer).value(width).value(height),
                          grid, 1, 1, 256, 1, 1);
            }
            sw.stop();
            CRT_CHECKED(crt_memcpy_d2h_async(device.ctx(), host_pixels.data(), pixel_buffer.data(), pixel_buffer.bytes()));
            device.synchronize();
            printf("frame %d kernel: %.3f ms\n", frame, sw.getMs());
            if (frame > 1) total_ms += sw.getMs();
        }
        if (frames > 1)
            printf("mean kernel time (frames 2..%d): %.3f ms = %.1f Mpix/s\n", frames, total_ms / (frames - 1),
                   (double)n * (frames - 1) / total_ms / 1e3);
        uint64_t h = 1469598103934665603ull;  // FNV-1a-64 of the RGBA8 image, for cross-checks with the Python host
        for (uint8_t b : host_pixels) h = (h ^ b) * 1099511628211ull;
        printf("rgba8 fnv1a64: %016llx\n", (unsigned long long)h);
        if (!out_ppm.empty())
        {
            FILE* f = fopen(out_ppm.c_str(), "wb");
            if (!f) throw crt::Error(CRT_EINVAL, "cannot write " + out_ppm);
            fprintf(f, "P6\n%d %d\n255\n", width, height);
            for (int y = height - 1; y >= 0; y--)  // buffers are bottom-up (10_restir_di.cu:18-20)
                for (int x = 0; x < width; x++) fwrite(&host_pixels[4 * ((size_t)y * width + x)], 1, 3, f);
            fclose(f);
        }
        if (!dump_accum.empty())
        {
            const std::vector<crt_float4> acc = accumulation_buffer.toHost();
            FILE* f = fopen(dump_accum.c_str(), "wb");
            if (!f) throw crt::Error(CRT_EINVAL, "cannot write " + dump_accum);
            fwrite(acc.data(), sizeof(crt_float4), acc.size(), f);
            fclose(f);
        }
        CRT_CHECKED(crt_destroy_geometry(device.ctx(), geom));
    }
    catch (const crt::Error& e)
    {
        fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
