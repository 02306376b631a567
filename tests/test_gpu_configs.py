"""GPU parity at the BASELINE configurations themselves (configs 2, 3, 4 at 1920x1080 on their own scenes and
cameras), the by-name launch layer, the C++ host above the C ABI, the reference GPU build as a pin for the
argument-evaluation order, and the frame fingerprint bench.py prints.

Bars as in test_gpu_parity.py: bit-exact in CRT_MATH_EXACT against the oracle (math mode 1) on bands of rows the oracle
computes in seconds; mean relative L1 <= 1e-3 (north star) for accumulated radiance in the default arithmetic."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import cedecrt
import orc
from helpers import DeviceAsOracle, reservoir_mismatch, same, scene, small_scene
from test_oracle_pinning import SURVEY_PRIMARY, pixel_classes, primary_goldens

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAM_AO = SURVEY_PRIMARY["blocks_ao"][0]
CAM_PT = SURVEY_PRIMARY["blocks_pt"][0]
CAM_RESTIR = SURVEY_PRIMARY["blocks_restir"][0]
CAM_CB = ((0.0, 2.7, 9.0), (0.0, 2.7, 0.0))
REL_L1_TOL = 1e-3
W, H = 1920, 1080


@pytest.fixture(scope="module")
def rt():
    r = cedecrt.Runtime(0)
    yield r
    r.close()


@pytest.fixture()
def exact(rt, port):
    rt.set_math_mode(cedecrt.MATH_EXACT)
    port.set_math_mode(1)
    yield DeviceAsOracle(rt)
    port.set_math_mode(0)
    port.set_example(9)
    port.set_range(0, -1)
    rt.set_math_mode(cedecrt.MATH_LIBDEVICE)


def band(y0, y1):
    return slice((H - y1) * W, (H - y0) * W)  # bottom-up storage (10_restir_di.cu:18-20)


# ------------------------------------------------------------------ primary visibility: the survey's goldens on the GPU
@pytest.mark.parametrize("name", sorted(SURVEY_PRIMARY))
def test_primary_visibility_survey_goldens(rt, name):
    """k_raycast on the three scenes of helpers.scene at the reference cameras, 1920x1080: pixel classes and the
    FNV-1a-64 of the primitive-id image equal the goldens of test_oracle_pinning.py (for blocks_ao the ones SURVEY.md
    section 4 extracted from the reference code; the oracle reproduces them on the CPU) — every one of 2 073 600 closest
    hits, ties included"""
    cam, classes, prim_hash, _ = primary_goldens(name)
    tris = scene(name)
    d_tris = rt.to_device(tris)
    g = rt.build_geometry(d_tris)
    vis = rt.buffer(cedecrt.VISIBILITY, W * H)
    rt.raycast(W, H, g, d_tris, cedecrt.lookat(*cam, W, H), vis)
    idx = vis.to_host()["index"]
    g.destroy()
    assert pixel_classes(idx, tris) == classes
    assert orc.fnv1a64(idx, orc.SURVEY_FNV_BASIS) == prim_hash


# ------------------------------------------------------------------ config 2: 06_ao_hiprt, blocks_ao, 32 AO rays
def test_config2_ao_1080p_band_bit_exact(exact, port):
    tris = scene("blocks_ao")
    port.set_example(6)
    g, gp = exact.geom_build(tris), port.geom_build(tris)
    mine = exact.ao(W, H, g, tris, exact.lookat(*CAM_AO, W, H), 32).reshape(-1, 4)
    y0, y1 = 508, 572
    port.set_range(y0 * W, y1 * W)
    ref = port.ao(W, H, gp, tris, port.lookat(*CAM_AO, W, H), 32).reshape(-1, 4)
    rows = band(y0, y1)
    assert same(mine[rows], ref[rows])
    assert len(np.unique(mine[rows][:, 0])) > 20  # a real AO gradient, not a constant
    # whole frame: background pixels are exactly the sky pixels of the primary-visibility golden
    assert int((mine[:, 0] == 32).sum()) >= SURVEY_PRIMARY["blocks_ao"][1][0]
    # rays the kernel counted: one primary per pixel + 32 per hit pixel (SURVEY.md section 8d)
    before = exact.rt.inline_rays_traced()
    exact.ao(W, H, g, tris, exact.lookat(*CAM_AO, W, H), 32)
    after = exact.rt.inline_rays_traced()
    assert after[0] - before[0] == W * H and after[1] - before[1] == 32 * SURVEY_PRIMARY["blocks_ao"][1][2]


# ------------------------------------------------------------------ config 3: 08_nee, blocks_pt, max depth 4
def test_config3_nee_1080p_band_bit_exact_two_frames(exact, port):
    tris = scene("blocks_pt")
    port.set_example(8)
    opt = orc.make_options(accumulate=1, max_depth=4)
    lights = orc.light_indices(tris)
    assert len(lights) == 72
    g, gp = exact.geom_build(tris), port.geom_build(tris)
    a, b = np.zeros((W * H, 4), np.float32), np.zeros((W * H, 4), np.float32)
    y0, y1 = 508, 572
    port.set_range(y0 * W, y1 * W)
    before = exact.rt.inline_rays_traced()
    for frame in (1, 2):
        port.path_trace(W, H, frame, gp, tris, lights, port.lookat(*CAM_PT, W, H), opt, a)
        exact.path_trace(8, W, H, frame, g, tris, lights, exact.lookat(*CAM_PT, W, H), opt, b)
    after = exact.rt.inline_rays_traced()
    rows = band(y0, y1)
    assert same(a[rows], b[rows]) and float(b[rows][:, :3].sum()) > 0 and (b[:, 3] == 2).all()
    # 08_nee traces one closest-hit ray per path vertex and one shadow ray per diffuse vertex (08_nee.cu:43,76-77):
    # between 1 and max_depth closest rays per pixel per frame, never more shadow rays than closest rays
    closest, shadow = after[0] - before[0], after[1] - before[1]
    assert 2 * W * H <= closest <= 2 * 4 * W * H and 0 < shadow <= closest


def test_config3_nee_64_frames_within_tolerance(rt, port):
    """64 accumulated frames, depth 4, default arithmetic of the per-kernel path against the oracle's libm arithmetic,
    at reduced size (the oracle runs every frame in full)"""
    tris = scene("blocks_pt")
    w, h, N = 320, 180, 64
    rt.set_math_mode(cedecrt.MATH_REFERENCE)
    port.set_math_mode(0)
    port.set_example(8)
    dev = DeviceAsOracle(rt)
    opt = orc.make_options(accumulate=1, max_depth=4)
    lights = orc.light_indices(tris)
    g, gp = dev.geom_build(tris), port.geom_build(tris)
    a, b = np.zeros((w * h, 4), np.float32), np.zeros((w * h, 4), np.float32)
    d_acc = rt.buffer(cedecrt.FLOAT4, w * h).zero()
    d_tris, d_lights = g.triangles, rt.to_device(lights)
    rg = cedecrt.lookat(*CAM_PT, w, h)
    for frame in range(1, N + 1):
        port.path_trace(w, h, frame, gp, tris, lights, port.lookat(*CAM_PT, w, h), opt, a)
        rt.path_trace(8, w, h, frame, g, d_tris, d_lights, rg, cedecrt.Options.from_numpy(opt), d_acc)
    b = d_acc.to_host().view(np.float32).reshape(-1, 4)
    port.set_example(9)
    assert (b[:, 3] == N).all() and np.isfinite(b).all()
    err = float(np.abs(a[:, :3] - b[:, :3]).sum() / np.abs(a[:, :3]).sum())
    print("08_nee, %d frames, mean relative L1 %.3e" % (N, err))
    assert err <= REL_L1_TOL


# ------------------------------------------------------------------ config 4: 09_ris, blocks_restir, shadowed target
def test_config4_ris_shadowed_1080p_band_bit_exact(exact, port):
    tris = scene("blocks_restir")
    port.set_example(9)
    opt = orc.make_options(accumulate=1, ris_sample_count=32, use_shadowed_target_function=1)
    lights = orc.light_indices(tris)
    assert len(lights) == 145344
    g, gp = exact.geom_build(tris), port.geom_build(tris)
    a, b = np.zeros((W * H, 4), np.float32), np.zeros((W * H, 4), np.float32)
    y0, y1 = 520, 584  # 35 rays per path vertex, depth up to 6: 64 rows keep the oracle at a few seconds
    port.set_range(y0 * W, y1 * W)
    port.path_trace(W, H, 1, gp, tris, lights, port.lookat(*CAM_RESTIR, W, H), opt, a)
    before, decided0 = exact.rt.inline_rays_traced(), exact.rt.rays_decided_at_emission()[1]
    exact.path_trace(9, W, H, 1, g, tris, lights, exact.lookat(*CAM_RESTIR, W, H), opt, b)
    after, decided = exact.rt.inline_rays_traced(), exact.rt.rays_decided_at_emission()[1] - decided0
    rows = band(y0, y1)
    assert same(a[rows], b[rows]) and float(b[rows][:, :3].sum()) > 0
    closest, walked = after[0] - before[0], after[1] - before[1]
    # the candidate rays that the triangle they start on stops are settled by the emitting kernel (crt_rays_decided_at_emission):
    # a light below the vertex's horizon (measured on this scene and camera: 9 % of the uniformly drawn candidates)
    assert 0.02 * (walked + decided) < decided < 0.5 * (walked + decided), (walked, decided)
    shadow = walked + decided
    # 32 candidates + the visibility ray per diffuse vertex (09_ris.cu:90-112); the final target function's ray (:116-119) repeats
    # the visibility ray's arguments and is not traced again by the wavefront form (34 per vertex with CRT_WAVEFRONT=0)
    assert shadow % 33 == 0 and shadow // 33 <= closest


# ------------------------------------------------------------------ Shader::launch shape for every kernel name
def test_launch_by_name_round_trips_every_kernel(rt):
    """crt_launch(name, void** params) (common/shader.hpp:179-199) against the typed exports, for all twelve names:
    a mis-unpacked by-value struct or a swapped slot shows up as a different buffer"""
    tris = small_scene("blocks_ao").copy()
    tris["emissive"][100:140] = (5.0, 4.0, 3.0)
    w, h = 96, 54
    rt.set_math_mode(cedecrt.MATH_LIBDEVICE)
    d_tris = rt.to_device(tris)
    d_lights = rt.to_device(cedecrt.light_indices(tris))
    g = rt.build_geometry(d_tris)
    rg = cedecrt.lookat(*CAM_AO, w, h)
    eye = cedecrt.Float3(*[float(np.float32(v)) for v in CAM_AO[0]])
    opt = cedecrt.Options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1, max_depth=3,
                          sky_color=(0.1, 0.2, 0.3))
    n = w * h

    def bufs():
        return dict(vis=rt.buffer(cedecrt.VISIBILITY, n), r0=rt.buffer(cedecrt.RESERVOIR, n).zero(),
                    r1=rt.buffer(cedecrt.RESERVOIR, n).zero(), tmp=rt.buffer(cedecrt.RESERVOIR, n).zero(),
                    acc=rt.buffer(cedecrt.FLOAT4, n).zero(), pix=rt.buffer(np.uint8, 4 * n).zero())

    A, B = bufs(), bufs()
    for frame in (1, 2):
        # typed exports
        rt.raycast(w, h, g, d_tris, rg, A["vis"])
        rt.generate_candidate(w, h, frame, g, d_tris, A["vis"], (eye.x, eye.y, eye.z), d_lights, opt, A["r0"])
        rt.temporal_resampling(w, h, frame, g, d_tris, A["vis"], (eye.x, eye.y, eye.z), opt, A["tmp"], A["r0"])
        rt.save_temporal_reservoir(w, h, A["r0"], A["tmp"])
        rt.spatial_resampling(w, h, frame, 0, g, d_tris, A["vis"], (eye.x, eye.y, eye.z), opt, A["r0"], A["r1"])
        rt.resolve(A["acc"], w, h, g, d_tris, A["vis"], (eye.x, eye.y, eye.z), opt, A["r1"])
        rt.tone_mapping(A["pix"], A["acc"], w, h)
        # the same through crt_launch, arguments in the reference's ShaderArgument order (10_restir_di.cpp:270-372)
        rt.launch("raycast", w, h, g, d_tris, rg, B["vis"])
        rt.launch("generate_candidate", w, h, frame, g, d_tris, B["vis"], eye, d_lights, opt, B["r0"])
        rt.launch("temporal_resampling", w, h, frame, g, d_tris, B["vis"], eye, opt, B["tmp"], B["r0"])
        rt.launch("save_temporal_reservoir", w, h, B["r0"], B["tmp"])
        rt.launch("spatial_resampling", w, h, frame, 0, g, d_tris, B["vis"], eye, opt, B["r0"], B["r1"])
        rt.launch("resolve", B["acc"], w, h, g, d_tris, B["vis"], eye, opt, B["r1"])
        rt.launch("tone_mapping", B["pix"], B["acc"], w, h)
    for k in A:
        assert same(A[k].to_host(), B[k].to_host()), k
    assert float(A["acc"].to_host().view(np.float32).reshape(-1, 4)[:, :3].sum()) > 0
    rt.clear(A["acc"], w, h)
    rt.launch("clear", B["acc"], w, h)
    assert same(A["acc"].to_host(), B["acc"].to_host()) and not A["acc"].to_host().view(np.uint8).any()
    # single-kernel examples
    for ex in (7, 8, 9):
        a, b = rt.buffer(cedecrt.FLOAT4, n).zero(), rt.buffer(cedecrt.FLOAT4, n).zero()
        for frame in (1, 2):
            rt.path_trace(ex, w, h, frame, g, d_tris, d_lights, rg, opt, a)
            if ex == 7:
                rt.launch("path_trace_07", w, h, frame, g, d_tris, rg, opt, b)
            else:
                rt.launch("path_trace_%02d" % ex, w, h, frame, g, d_tris, d_lights, rg, opt, b)
        assert same(a.to_host(), b.to_host()), ex
        assert float(a.to_host().view(np.float32).reshape(-1, 4)[:, :3].sum()) > 0, ex
    p1, p2 = rt.buffer(np.uint8, 4 * n).zero(), rt.buffer(np.uint8, 4 * n).zero()
    rt.ao(p1, rg, w, h, g, d_tris, 16)
    rt.launch("ao_06", p2, rg, w, h, g, d_tris, 16)
    assert same(p1.to_host(), p2.to_host()) and len(np.unique(p1.to_host())) > 5
    g.destroy()


# ------------------------------------------------------------------ the C++ host above the C ABI
def test_headless_cpp_host_matches_the_ctypes_path(rt, tmp_path):
    """cedec-2024-rt_b200/restir_di_headless — the reference's application loop in C++ (TypedBuffer, Shader::launch ->
    crt_launch for the nine kernel names of the frame, Stopwatch; host/crt_host.hpp) — renders the same frames as the
    Python host does through ctypes: accumulation bit for bit, in launch-list mode and with --fused"""
    exe = os.path.join(ROOT, "cedec-2024-rt_b200", "restir_di_headless")
    tris = scene("blocks_restir")
    tri_file = str(tmp_path / "blocks_restir.tri")
    tris.tofile(tri_file)
    w, h, frames = 480, 270, 3
    kw = dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    for fused in (False, True):
        out = str(tmp_path / ("acc_%d.f32" % fused))
        cmd = [exe, "--scene", tri_file, "--size", str(w), str(h), "--frames", str(frames), "--dump-accum", out]
        r = subprocess.run(cmd + (["--fused"] if fused else []), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, (r.stdout[-1000:], r.stderr[-2000:])
        assert "lights: 145344" in r.stdout and "mean kernel time" in r.stdout
        theirs = np.fromfile(out, np.float32).reshape(-1, 4)
        # the C++ host leaves the library's default arithmetic (CRT_MATH_REFERENCE): so does this context
        rt.set_math_mode(cedecrt.MATH_REFERENCE)
        app = cedecrt.RestirDI(rt, w, h, tris, *CAM_RESTIR, cedecrt.Options(**kw), fused=fused)
        for _ in range(frames):
            app.frame()
        mine = app.accumulation.to_host().view(np.float32).reshape(-1, 4)
        assert same(mine, theirs), "fused" if fused else "launch list"
        line = [l for l in r.stdout.splitlines() if l.startswith("rgba8 fnv1a64")][0]
        pix = app.pixels.to_host()
        assert line.split()[-1] == orc.fnv1a64(pix, orc.SURVEY_FNV_BASIS)  # the host prints the survey-style hash
    rt.set_math_mode(cedecrt.MATH_LIBDEVICE)


# ------------------------------------------------------------------ the reference's own GPU build as a pin
def run_ref_gpu(args, timeout=600):
    bin_dir = os.path.join(ROOT, "baseline", "_ref", "bin")
    exe = os.path.join(bin_dir, "ref_gpu")
    if not os.path.exists(exe):
        pytest.skip("baseline/_ref/bin/ref_gpu not staged (make -C oracle refgpu, needs the reference checkout)")
    env = dict(os.environ, LD_LIBRARY_PATH=bin_dir + ":/usr/local/cuda/lib64:" + os.environ.get("LD_LIBRARY_PATH", ""))
    r = subprocess.run([exe, "--base", "../"] + args, cwd=bin_dir, env=env, capture_output=True, text=True, timeout=timeout)
    line = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if not line or "unavailable" in json.loads(line[-1]):
        pytest.skip("the reference HIPRT build does not run here: %s" % (line[-1] if line else r.stderr[-300:]))
    return json.loads(line[-1])


def test_reference_gpu_build_pins_the_argument_order(port, tmp_path):
    """The port (and the CUDA path) draw the randoms of sample_light(..., uniformf(), uniformf(), uniformf())
    (10_restir_di.cu:88-90) left to right; the reference compiled by g++ (oracle/_ref) draws them right to left.  Which
    one the reference's real GPU build does is decided here by that build itself: its Reservoir[] straight after
    generate_candidate on frame 1 (cornellbox1, 96x54) against the port in both orders, fed with the GPU build's own
    Visibility so that HIPRT's intersector does not enter the comparison."""
    tris = small_scene("cornellbox1")
    w, h = 96, 54
    tri_file, dump = str(tmp_path / "cb.tri"), str(tmp_path / "cand.bin")
    tris.tofile(tri_file)
    run_ref_gpu(["--tri", tri_file, "--width", str(w), "--height", str(h), "--frames", "1", "--warmup", "0",
                 "--eye", "0", "2.7", "9", "--lookat", "0", "2.7", "0", "--dump-candidates", dump])
    raw = np.fromfile(dump, np.uint8)
    n = w * h
    ref = raw[:n * 76].view(orc.RESERVOIR)
    vis = raw[n * 76:].view(orc.VISIBILITY).copy()
    assert len(vis) == n and int((vis["index"] >= 0).sum()) > 1000
    g = port.geom_build(tris)
    lights = orc.light_indices(tris)
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    port.set_math_mode(0)
    em = (tris["emissive"] > 0).any(1)
    diffuse = (vis["index"] >= 0)
    diffuse[diffuse] = ~em[vis["index"][diffuse]]
    match = {}
    try:
        for order in (0, 1):
            port.set_arg_order(order)
            mine = port.generate_candidate(w, h, 1, g, tris, vis, CAM_CB[0], lights, opt)
            close = np.abs(mine["hit_position"] - ref["hit_position"]).max(1) < 1e-3
            match[order] = float((close & (mine["M"] == ref["M"]))[diffuse].mean())
    finally:
        port.set_arg_order(0)
    print("selected light sample equal to the reference GPU build's: left-to-right %.4f, right-to-left %.4f" % (match[0], match[1]))
    assert match[0] > 0.98 and match[1] < 0.5


# ------------------------------------------------------------------ temporal reprojection (extension, SURVEY section 8 f2)
def test_temporal_reprojection_bit_exact_with_a_moving_camera(rt, exact, port):
    """crt_temporal_resampling_reprojected against its specification (oracle/port: reproject_pixel): the chain with two
    camera moves on blocks_restir at 480x270, exact arithmetic — stage outputs and accumulation bit for bit; the resident
    host loop (cedecrt.RestirDI(reproject=True).set_camera) gives the same frames; and by name through crt_launch"""
    from test_reprojection import KW, moved_camera_chain

    tris = small_scene("blocks_ao").copy()
    tris["emissive"][100:140] = (5.0, 4.0, 3.0)
    w, h = 128, 72
    a = moved_camera_chain(port, tris, w, h, 1, True)
    b = moved_camera_chain(exact, tris, w, h, 1, True)
    rt.set_math_mode(cedecrt.MATH_EXACT)
    port.set_math_mode(1)
    assert same(a.vis["index"], b.vis["index"]) and same(a.vis["uv"], b.vis["uv"])
    assert reservoir_mismatch(a.temporal, b.temporal) == 0 and reservoir_mismatch(a.out, b.out) == 0
    assert same(a.accum, b.accum) and float(a.accum[:, :3].sum()) > 0
    # the resident loop
    app = cedecrt.RestirDI(rt, w, h, tris, *CAM_AO, cedecrt.Options(**KW), reproject=True)
    for _ in range(2):
        app.frame()
    app.set_camera((8.4, 7.8, 8.1), (0.1, 0.0, -0.1))
    app.frame()
    prev_rg = cedecrt.RayGenerator.from_buffer_copy(bytes(app.prev_raygen))
    app.set_camera((8.9, 7.5, 8.3), (0.2, 0.1, -0.2))
    app.frame()
    assert same(app.accumulation.to_host().view(np.float32).reshape(-1, 4), a.accum)
    assert reservoir_mismatch(app.temporal.to_host(), a.temporal) == 0
    # by name: frame 4's temporal step again, from the same inputs
    n = w * h
    cand = rt.buffer(cedecrt.RESERVOIR, n)
    eye = cedecrt.Float3(*app.eye)
    rt.generate_candidate(w, h, 4, app.geom, app.triangles, app.visibility, app.eye, app.lights, app.options, cand)
    one, two = rt.to_device(cand.to_host()), rt.to_device(cand.to_host())
    hist = rt.to_device(a.temporal)  # any history will do: both calls read the same
    rt.temporal_resampling_reprojected(w, h, 4, app.geom, app.triangles, app.visibility, app.eye, app.options, prev_rg, hist, one)
    rt.launch("temporal_resampling_reprojected", w, h, 4, app.geom, app.triangles, app.visibility, eye, app.options, prev_rg, hist, two)
    assert same(one.to_host(), two.to_host())
    with pytest.raises(cedecrt.CrtError, match="in place"):
        rt.temporal_resampling_reprojected(w, h, 4, app.geom, app.triangles, app.visibility, app.eye, app.options, prev_rg, one, one)
    # the fused frame with the same look-up (crt_restir_set_previous_camera): the same frames, bit for bit — and with options
    # that take the per-kernel path inside crt_restir_di_frame (the shadowed target function) against the launch list
    fused = cedecrt.RestirDI(rt, w, h, tris, *CAM_AO, cedecrt.Options(**KW), fused=True, reproject=True)
    for _ in range(2):
        fused.frame()
    fused.set_camera((8.4, 7.8, 8.1), (0.1, 0.0, -0.1))
    fused.frame()
    fused.set_camera((8.9, 7.5, 8.3), (0.2, 0.1, -0.2))
    fused.frame()
    assert same(fused.accumulation.to_host().view(np.float32).reshape(-1, 4), a.accum)
    d = a.vis["index"] >= 0
    d[d] = ~(tris["emissive"] > 0).any(1)[a.vis["index"][d]]
    assert reservoir_mismatch(fused.export_aos(fused.temporal)[d], a.temporal[d]) == 0
    assert reservoir_mismatch(fused.output_reservoirs()[d], a.out[d]) == 0
    assert same(fused.pixels.to_host(), app.pixels.to_host())
    kw_sh = dict(KW, use_shadowed_target_function=1, ris_sample_count=4)
    x = cedecrt.RestirDI(rt, w, h, tris, *CAM_AO, cedecrt.Options(**kw_sh), fused=True, reproject=True)
    y = cedecrt.RestirDI(rt, w, h, tris, *CAM_AO, cedecrt.Options(**kw_sh), fused=False, reproject=True)
    for app2 in (x, y):
        app2.frame()
        app2.set_camera((8.4, 7.8, 8.1), (0.1, 0.0, -0.1))
        app2.frame()
    assert same(x.accumulation.to_host(), y.accumulation.to_host()) and same(x.temporal.to_host(), y.temporal.to_host())
    # a context that renders a row range may look history up as well: the host then provides the other rows of `temporal`
    # (tests/gpu_slab_worker.py, modes *_reproject: N slabs == 1 slab); only the direct-store slab links are refused
    rt.set_row_range(8, 40)
    try:
        fused.frame()
    finally:
        rt.set_row_range(0, -1)
        rt.restir_set_previous_camera(None)


# ------------------------------------------------------------------ frame overlap
def test_frame_overlap_changes_no_bit():
    """crt_set_frame_overlap: the tail of every frame (resolve rays + tone mapping) on a second stream, beside the next
    frame's raycast / candidate kernels — accumulation, RGBA8 and final reservoirs stay what the serial frames give"""
    tris = scene("blocks_restir")
    w, h, frames = 960, 540, 5
    kw = dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    serial, lapped = cedecrt.Runtime(0), cedecrt.Runtime(0)
    lapped.set_frame_overlap(True)
    a = cedecrt.RestirDI(serial, w, h, tris, *CAM_RESTIR, cedecrt.Options(**kw), fused=True)
    b = cedecrt.RestirDI(lapped, w, h, tris, *CAM_RESTIR, cedecrt.Options(**kw), fused=True)
    b.prefetch = True  # and the next frame's primary rays traced ahead of time on a third stream
    launches = lapped.launch_count(), serial.launch_count()
    for f in range(frames):
        a.frame()
        b.frame()
        if f == 2:  # a read in the middle of the sequence must see the finished frame too
            assert same(a.pixels.to_host(), b.pixels.to_host())
    assert same(a.accumulation.to_host(), b.accumulation.to_host())
    assert same(a.pixels.to_host(), b.pixels.to_host())
    assert reservoir_mismatch(a.output_reservoirs(), b.output_reservoirs()) == 0
    assert serial.shadow_rays_traced() == lapped.shadow_rays_traced()
    assert same(a.visibility.to_host(), b.visibility.to_host())
    # frames 2.. took their Visibility rows from the prefetch: one raycast launch per frame all the same (frames + 1 with the
    # last prefetch), never two
    assert lapped.launch_count() - launches[0] == serial.launch_count() - launches[1] + 1
    # a camera the prefetch did not anticipate: the frame traces its own rays, the stale prefetch is dropped
    a.set_camera((-0.3, 22.3, -6.4), (5.2, 20.8, 1.4))
    b.set_camera((-0.3, 22.3, -6.4), (5.2, 20.8, 1.4))
    a.frame()
    b.frame()
    assert same(a.visibility.to_host(), b.visibility.to_host()) and same(a.accumulation.to_host(), b.accumulation.to_host())
    assert float(a.accumulation.to_host().view(np.float32).reshape(-1, 4)[:, :3].sum()) > 0
    serial.close()
    lapped.close()


# ------------------------------------------------------------------ bench.py's frame fingerprint
def test_bench_frame_hash(rt):
    """the frame_hash of bench.py's JSON line (config 5 at 4K, exact arithmetic, frames 1-2): deterministic, equal for
    one slab and for three slabs on one GPU (what SCALE compares across 1, 2, 4, 8 GPUs), and equal to the committed
    value (tests/golden/frame_hash.json) — which the full-size band test ties to the oracle bit for bit"""
    import torch

    sys.path.insert(0, ROOT)
    import bench
    import slabs

    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    tris, cam, _ = bench.load_workload()
    torch.cuda.set_device(0)
    with torch.cuda.stream(torch.cuda.Stream()):
        one = slabs.SlabRenderer(torch, None, 0, 1, tris, cam, 3840, 2160, fused=True)
        h1 = bench.frame_hash(torch, None, one, 1)
        h1b = bench.frame_hash(torch, None, one, 1)
        assert h1["value"] == h1b["value"]
        del one
        group = slabs.SlabGroup(torch, None, 0, 1, tris, cam, 3840, 2160, sub=3)
        h3 = bench.frame_hash(torch, None, group, 1)
        group.close()
    assert h1["value"] == h3["value"]
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "frame_hash.json")))
    key = "config5_4k" if len(tris) == 9590208 else "procedural_4k"  # the staged scene or bench.py's stand-in
    print("frame_hash", h1["value"], "golden", golden[key])
    assert h1["value"] == golden[key]


# ------------------------------------------------------------------ pipelined read-back (bench.py's e2e loop)
def test_pipelined_readback_delivers_every_frame(rt):
    """SlabRenderer.download_pixels_async: frame i's RGBA8 image travels on a copy stream while frame i+1 renders, the
    frames alternating between two device images.  Every delivered image must equal the one the reference's read-back
    (copy on the frame's stream, then synchronise: 10_restir_di.cpp:386-389) delivers for the same frame, with and
    without frame overlap."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench
    import slabs

    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    tris, cam, _ = bench.load_workload()
    torch.cuda.set_device(0)
    W, H, frames = 960, 544, 5
    with torch.cuda.stream(torch.cuda.Stream()):
        ref = slabs.SlabRenderer(torch, None, 0, 1, tris, cam, W, H, fused=True)
        want = []
        for _ in range(frames):
            ref.frame()
            ref.download_pixels()
            ref.stream.synchronize()
            want.append(ref.host_pixels.numpy().copy())
        ref.close()
        assert any(not np.array_equal(want[0], w) for w in want[1:])  # the accumulated image changes from frame to frame
        for overlap in (False, True):
            r = slabs.SlabRenderer(torch, None, 0, 1, tris, cam, W, H, fused=True, overlap=overlap)
            got, prev = [], None
            for _ in range(frames):
                r.frame()
                slot = r.download_pixels_async()
                if prev is not None:
                    got.append(r.wait_download(prev).numpy().copy())
                prev = slot
            got.append(r.wait_download(prev).numpy().copy())
            r.join()
            r.close()
            for i in range(frames):
                assert np.array_equal(got[i], want[i]), (overlap, i)
