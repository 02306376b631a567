"""Parity tests proper: the CUDA kernels, called through the C ABI (libcedecrt.so via ctypes), against the
CPU oracle (oracle/port, pinned to the reference by test_oracle_pinning.py) on the same seeded inputs.

Bars (north star + tier rules):
  * index / byte / integer work — primitive ids, uv bits, RGBA8, M — bit-exact.  With CRT_MATH_EXACT the whole
    ReSTIR chain is bit-exact, stage by stage, because every float op then rounds exactly like the oracle's.
  * default math (CUDA libdevice float functions, what the reference's NVRTC build computes): accumulated
    radiance within mean relative L1 <= 1e-3 of the oracle (tolerance from BASELINE.json's north star).
  * full-size inputs: size-independent properties (BVH == exhaustive search on the GPU, determinism,
    pixel-class counts, untouched sky/emissive reservoirs).
"""
import os

import numpy as np
import pytest

import cedecrt
import orc
from helpers import DeviceAsOracle, reservoir_mismatch, same, scene, small_scene

pytestmark = pytest.mark.gpu

CAM_CB = ((0.0, 2.7, 9.0), (0.0, 2.7, 0.0))
CAM_AO = ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0))
CAM_RESTIR = ((-0.579885, 22.194597, -6.567105), (5.224952, 20.847435, 1.431192))  # 10_restir_di.cpp:188-189
REL_L1_TOL = 1e-3  # BASELINE.json north star: "mean relative L1 <= 1e-3"


@pytest.fixture(scope="module")
def rt():
    import cedecrt

    r = cedecrt.Runtime(0)
    yield r
    r.close()


@pytest.fixture()
def dev(rt):
    import cedecrt

    rt.set_math_mode(cedecrt.MATH_LIBDEVICE)
    return DeviceAsOracle(rt)


def lit_blocks_ao():
    t = small_scene("blocks_ao").copy()
    t["emissive"][100:140] = (5.0, 4.0, 3.0)
    return t


def config5():
    """the scene and camera bench.py renders (bench.load_workload)"""
    import bench

    tris, cam, _ = bench.load_workload()
    return tris, cam


def rel_l1(a, b):
    ra, rb = a[:, :3] / a[:, 3:4], b[:, :3] / b[:, 3:4]
    return float(np.abs(ra - rb).sum() / np.abs(rb).sum())


# ------------------------------------------------------------------ traversal
def test_refit_equals_exhaustive_search_and_rebuild(rt):
    """crt_refit_geometry after vertices moved on the device: closest hits equal the exhaustive loop's and a fresh
    build's on random rays (blocks_restir, 1.6 M triangles); refit time is reported next to build time"""
    tris = scene("blocks_restir").copy()
    d_tris = rt.to_device(tris)
    geom = rt.build_geometry(d_tris)
    rng = np.random.default_rng(9)
    tris["vertices"][100000:400000] += rng.uniform(-2.0, 2.0, 3).astype(np.float32)
    tris["vertices"][900000:900500] += rng.uniform(-0.1, 0.1, (500, 3, 3)).astype(np.float32)
    tris["vertices"][:36] += np.float32(40.0)  # the scene box grows
    d_tris.upload(tris)
    geom.refit()
    st = geom.stats()
    assert st["refit_ms"] > 0  # typically 1.4 ms against an 18 ms build; a first call also pays for allocations
    lo, hi = tris["vertices"].reshape(-1, 3).min(0), tris["vertices"].reshape(-1, 3).max(0)
    n = 4096
    org = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    dirs = rng.standard_normal((n, 3)).astype(np.float32)
    p_refit, tuv_refit = rt.trace_closest(geom, org, dirs)
    fresh = rt.build_geometry(d_tris)
    p_fresh, tuv_fresh = rt.trace_closest(fresh, org, dirs)
    assert same(p_refit, p_fresh) and same(tuv_refit, tuv_fresh)
    m = 256
    p_brute, tuv_brute = rt.trace_closest(geom, org[:m], dirs[:m], brute=True)
    assert same(p_refit[:m], p_brute) and same(tuv_refit[:m], tuv_brute)
    assert (p_refit >= 0).sum() > n // 4
    print("refit %.2f ms, build %.2f ms (1.6 M triangles)" % (st["refit_ms"], st["build_ms"]))
    fresh.destroy()
    geom.destroy()


@pytest.mark.parametrize("scene", ["cornellbox1", "blocks_ao"])
def test_bvh_equals_exhaustive_search_small(rt, scene):
    tris = small_scene(scene)
    d_tris = rt.to_device(tris)
    g = rt.build_geometry(d_tris)
    rng = np.random.default_rng(3)
    n = 20000
    o = rng.uniform(-7, 7, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d[::5, 0] = 0.0
    d[1::7, 1] = 0.0
    o[::9] = np.round(o[::9])
    p1, t1 = rt.trace_closest(g, o, d)
    p2, t2 = rt.trace_closest(g, o, d, brute=True)
    assert same(p1, p2) and same(t1, t2)
    assert (p1 >= 0).sum() > n // 10
    a1 = rt.trace_any(g, o, d, 0.0, 5.0)
    p3, _ = rt.trace_closest(g, o, d, 0.0, 5.0, brute=True)
    assert same(a1, (p3 >= 0).astype(np.int32))
    g.destroy()


def test_bvh_equals_exhaustive_search_blocks_restir(rt):
    tris = scene("blocks_restir")
    d_tris = rt.to_device(tris)
    g = rt.build_geometry(d_tris)
    st = g.stats()
    assert st["n_tris"] == len(tris) and st["max_depth"] <= 48
    rng = np.random.default_rng(5)
    n = 4096
    eye = np.array(CAM_RESTIR[0], np.float32)
    o = (eye + rng.uniform(-20, 20, (n, 3))).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    p1, t1 = rt.trace_closest(g, o, d)
    p2, t2 = rt.trace_closest(g, o, d, brute=True)
    assert same(p1, p2) and same(t1, t2)
    assert (p1 >= 0).sum() > n // 4
    g.destroy()


@pytest.mark.parametrize("scene,cam,size", [("cornellbox1", CAM_CB, (96, 54)), ("blocks_ao", CAM_AO, (320, 180))])
def test_raycast_bit_exact(dev, port, scene, cam, size):
    tris = small_scene(scene)
    W, H = size
    outs = []
    for o in (port, dev):
        g = o.geom_build(tris)
        outs.append(o.raycast(W, H, g, tris, o.lookat(*cam, W, H)))
        o.geom_free(g)
    assert same(outs[0]["index"], outs[1]["index"]) and same(outs[0]["uv"], outs[1]["uv"])
    assert (outs[1]["_pad"] == 0).all()


def test_raycast_is_the_oracle_s_whatever_the_buffer_held(dev, port):
    """crt_raycast seeds each pixel's walk with the triangle its Visibility record names before the call (px_raycast_hinted):
    the result does not depend on it — own answers, another camera's, random ids, -1, garbage, the smaller id of a duplicate"""
    tris = small_scene("blocks_ao").copy()
    tris = np.concatenate([tris, tris[500:700]])
    W, H = 320, 180
    g, gp = dev.geom_build(tris), port.geom_build(tris)
    rt, c = dev.rt, dev.c
    rng = np.random.default_rng(5)
    rg0, rg1 = dev.lookat(*CAM_AO, W, H), dev.lookat((7.0, 9.0, 8.5), (0.5, 0.0, -0.5), W, H)
    want = [port.raycast(W, H, gp, tris, port.lookat(*CAM_AO, W, H)), port.raycast(W, H, gp, tris, port.lookat((7.0, 9.0, 8.5), (0.5, 0.0, -0.5), W, H))]
    n = len(tris)
    assert (want[0]["index"] >= n - 200).sum() > 0
    hint_sets = {
        "own answer": want[0]["index"].copy(),
        "other camera's answer": want[1]["index"].copy(),
        "random triangles": rng.integers(0, n, W * H).astype(np.int32),
        "none": np.full(W * H, -1, np.int32),
        "garbage": rng.integers(-2**31, 2**31 - 1, W * H).astype(np.int32),
        "the duplicate with the smaller id": np.where(want[0]["index"] >= n - 200, want[0]["index"] - (n - 200) + 500, want[0]["index"]).astype(np.int32),
    }
    for name, hints in hint_sets.items():
        for k, rg in enumerate((rg0, rg1)):
            vis = np.zeros(W * H, c.VISIBILITY)
            vis["index"] = hints
            d = rt.to_device(vis)
            rt.raycast(W, H, g, g.triangles, dev._rg(rg), d)
            got = d.to_host()
            assert same(got["index"], want[k]["index"]) and same(got["uv"], want[k]["uv"]), name
    dev.geom_free(g)
    port.geom_free(gp)


def test_raycast_blocks_restir_1080p_pixel_classes(dev, port):
    """config 4/5 camera on the blocks_restir stand-in: bit-exact primitive ids against the oracle on a band of rows, and
    the pixel-class counts of the whole frame"""
    tris = scene("blocks_restir")
    W, H = 1920, 1080
    g = dev.geom_build(tris)
    vis = dev.raycast(W, H, g, tris, dev.lookat(*CAM_RESTIR, W, H))
    idx = vis["index"]
    em = (tris["emissive"] > 0).any(1)
    sky = int((idx < 0).sum())
    emi = int(em[idx[idx >= 0]].sum())
    assert (sky, emi, W * H - sky - emi) == (292082, 47253, 1734265)
    gp = port.geom_build(tris)
    y0, y1 = 500, 564  # 64 rows of the oracle: seconds on a few cores
    port.set_range(y0 * W, y1 * W)
    ref = port.raycast(W, H, gp, tris, port.lookat(*CAM_RESTIR, W, H))
    port.set_range(0, -1)
    rows = slice((H - y1) * W, (H - y0) * W)  # bottom-up storage
    assert same(vis["index"][rows], ref["index"][rows]) and same(vis["uv"][rows], ref["uv"][rows])
    dev.geom_free(g)
    port.geom_free(gp)


# ------------------------------------------------------------------ ReSTIR chain
@pytest.mark.parametrize("scene", ["cornellbox1", "blocks_ao_lit"])
def test_restir_chain_bit_exact_in_exact_math_mode(dev, port, scene):
    import cedecrt

    tris = small_scene("cornellbox1") if scene == "cornellbox1" else lit_blocks_ao()
    cam, (W, H) = (CAM_CB, (96, 54)) if scene == "cornellbox1" else (CAM_AO, (160, 90))
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    port.set_math_mode(1)
    dev.set_math_mode(cedecrt.MATH_EXACT)
    chains = []
    for o in (port, dev):
        g = o.geom_build(tris)
        chains.append(orc.RestirChain(o, W, H, tris, g, *cam, opt))
    for frame in range(3):
        for ch in chains:
            ch.step()
        a, b = chains
        assert same(a.vis["index"], b.vis["index"]) and same(a.vis["uv"], b.vis["uv"])
        for name in ("buf0", "buf1", "temporal"):
            assert reservoir_mismatch(getattr(a, name), getattr(b, name)) == 0, (frame, name)
        assert same(a.accum, b.accum), frame
    pa = port.tone_mapping(chains[0].accum, W, H)
    pb = dev.tone_mapping(chains[1].accum, W, H)
    assert same(pa, pb)
    port.set_math_mode(0)


def test_restir_options_bit_exact(dev, port):
    import cedecrt

    tris = small_scene("cornellbox1")
    W, H = 64, 36
    port.set_math_mode(1)
    dev.set_math_mode(cedecrt.MATH_EXACT)
    for kw in (dict(use_shadowed_target_function=1, use_visibility_reuse=0, use_temporal_resampling=1,
                    use_spatial_resampling=1, ris_sample_count=8, spatial_resampling_passes=2),
               dict(use_spatial_resampling=0, use_temporal_resampling=1),
               dict(use_spatial_resampling=1, use_temporal_resampling=0, spatial_resampling_radius=5.0,
                    spatial_resampling_sample_count=2, accumulate=1)):
        opt = orc.make_options(**kw)
        outs = []
        for o in (port, dev):
            g = o.geom_build(tris)
            ch = orc.RestirChain(o, W, H, tris, g, *CAM_CB, opt)
            ch.step()
            ch.step()
            outs.append((ch.buf0.copy(), ch.buf1.copy(), ch.accum.copy()))
        assert reservoir_mismatch(outs[0][0], outs[1][0]) == 0 and reservoir_mismatch(outs[0][1], outs[1][1]) == 0
        assert same(outs[0][2], outs[1][2]), kw
    port.set_math_mode(0)


def test_restir_default_math_within_tolerance(rt, port):
    """default (libdevice) math: N accumulated frames of the resident frame loop vs the oracle (glibc math)"""
    import cedecrt

    tris = lit_blocks_ao()
    W, H, N = 160, 90, 8
    rt.set_math_mode(cedecrt.MATH_LIBDEVICE)
    app = cedecrt.RestirDI(rt, W, H, tris, *CAM_AO, cedecrt.Options(accumulate=1, use_temporal_resampling=1,
                                                                   use_spatial_resampling=1))
    g = port.geom_build(tris)
    ch = orc.RestirChain(port, W, H, tris, g, *CAM_AO,
                         orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1))
    for _ in range(N):
        app.frame()
        ch.step()
    acc = app.accumulation.to_host().view(np.float32).reshape(-1, 4)
    assert same(acc[:, 3], ch.accum[:, 3])
    err = rel_l1(acc, ch.accum)
    print("mean relative L1 after %d frames: %.3e" % (N, err))
    assert err <= REL_L1_TOL
    # generate_candidate has no transcendental: its output is bit-exact in every math mode
    vis = app.visibility.to_host()
    assert same(vis["index"], ch.vis["index"])


def test_fast_math_mode_within_tolerance_over_64_frames(rt, port):
    """The contracted-arithmetic modes of the fused frame — CRT_MATH_REFERENCE (the default: FMA contraction, IEEE
    division / square root, libdevice functions = the reference's own NVRTC arithmetic) and CRT_MATH_FAST (approximate
    division, hardware transcendentals) — with rays and triangle tests exact in both: 64 accumulated frames of blocks_ao
    with 40 emissive triangles at its own camera against the oracle.  Bars: primitive ids bit-exact; accumulated radiance
    within the north star's mean relative L1 <= 1e-3; the uncontracted LIBDEVICE mode on the same run stays below 1e-6.
    The bars were set on the config-4/5 scene and camera (blocks_restir, FAST 6e-5: profiles/r1/long_horizon_parity.txt),
    which the repository does not hold.  Its procedural stand-in (helpers.STAND_INS) at the config-4/5 camera does not
    meet them: on a B200, FAST 1.35e-3, REFERENCE 5.2e-6, LIBDEVICE 3.9e-6.  Stage by stage from the oracle's state of one
    frame (test_gpu_math_modes.py, 16 rows of the stand-in) FAST's stages match REFERENCE's, so no single stage shows a
    bias there; that the gap builds up across frames of FAST's own history is a hypothesis, not traced."""
    tris = lit_blocks_ao()
    W, H, N = 480, 270, 64
    kw = dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    g = port.geom_build(tris)
    ch = orc.RestirChain(port, W, H, tris, g, *CAM_AO, orc.make_options(**kw))
    apps = {}
    try:
        for mode in (cedecrt.MATH_FAST, cedecrt.MATH_REFERENCE, cedecrt.MATH_LIBDEVICE):
            rt.set_math_mode(mode)
            apps[mode] = cedecrt.RestirDI(rt, W, H, tris, *CAM_AO, cedecrt.Options(**kw), fused=True)
        for _ in range(N):
            ch.step()
            for mode, app in apps.items():
                rt.set_math_mode(mode)
                app.frame()
        err = {}
        for mode, app in apps.items():
            acc = app.accumulation.to_host().view(np.float32).reshape(-1, 4)
            assert same(app.visibility.to_host()["index"], ch.vis["index"])
            assert same(acc[:, 3], ch.accum[:, 3]) and np.isfinite(acc).all()
            err[mode] = rel_l1(acc, ch.accum)
        print("mean relative L1 after %d frames: fast %.3e, reference %.3e, libdevice %.3e" % (
            N, err[cedecrt.MATH_FAST], err[cedecrt.MATH_REFERENCE], err[cedecrt.MATH_LIBDEVICE]))
        assert err[cedecrt.MATH_FAST] <= REL_L1_TOL
        assert err[cedecrt.MATH_REFERENCE] <= REL_L1_TOL
        assert err[cedecrt.MATH_LIBDEVICE] <= 1e-6
    finally:
        rt.set_math_mode(cedecrt.MATH_LIBDEVICE)
        port.geom_free(g)


def test_generate_candidate_bit_exact_on_blocks_restir_band(dev, port):
    """the 32-candidate RIS loop + visibility-reuse shadow ray on the 1.6 M-triangle / 145 k-light blocks_restir stand-in"""
    tris = scene("blocks_restir")
    W, H = 1920, 1080
    lights = orc.light_indices(tris)
    assert len(lights) == 145344
    opt = orc.make_options()
    g, gp = dev.geom_build(tris), port.geom_build(tris)
    vis = dev.raycast(W, H, g, tris, dev.lookat(*CAM_RESTIR, W, H))
    res = dev.generate_candidate(W, H, 1, g, tris, vis, CAM_RESTIR[0], lights, opt)
    y0, y1 = 600, 616
    port.set_range(y0 * W, y1 * W)
    ref = np.zeros(W * H, orc.RESERVOIR)
    port.generate_candidate(W, H, 1, gp, tris, vis, CAM_RESTIR[0], lights, opt, ref)
    port.set_range(0, -1)
    rows = slice((H - y1) * W, (H - y0) * W)
    assert reservoir_mismatch(res[rows], ref[rows]) == 0
    assert (res[rows]["M"] == 32).sum() > 1000


# ------------------------------------------------------------------ examples 06-09
@pytest.mark.parametrize("ex", [7, 8, 9])
def test_path_tracers_bit_exact(dev, port, ex):
    import cedecrt

    tris = small_scene("cornellbox1")
    W, H = 64, 36
    opt = orc.make_options(accumulate=1, max_depth=4, ris_sample_count=8, sky_color=(0.1, 0.2, 0.3))
    lights = orc.light_indices(tris)
    port.set_math_mode(1)
    dev.set_math_mode(cedecrt.MATH_EXACT)
    port.set_example(ex)
    gp, g = port.geom_build(tris), dev.geom_build(tris)
    a, b = np.zeros((W * H, 4), np.float32), np.zeros((W * H, 4), np.float32)
    for frame in (1, 2):
        port.path_trace(W, H, frame, gp, tris, lights, port.lookat(*CAM_CB, W, H), opt, a)
        dev.path_trace(ex, W, H, frame, g, tris, lights, dev.lookat(*CAM_CB, W, H), opt, b)
    port.set_example(9)
    port.set_math_mode(0)
    assert same(a, b) and float(a[:, :3].sum()) > 0


def test_ao06_bit_exact(dev, port):
    import cedecrt

    tris = small_scene("blocks_ao")
    W, H = 160, 90
    port.set_math_mode(1)
    dev.set_math_mode(cedecrt.MATH_EXACT)
    port.set_example(6)
    gp, g = port.geom_build(tris), dev.geom_build(tris)
    a = port.ao(W, H, gp, tris, port.lookat(*CAM_AO, W, H), 32)
    b = dev.ao(W, H, g, tris, dev.lookat(*CAM_AO, W, H), 32)
    port.set_example(9)
    port.set_math_mode(0)
    assert same(a, b)


def test_launch_by_name_matches_direct_call(rt):
    """Shader::launch call shape (crt_launch) == the typed exports"""
    import ctypes as C

    import cedecrt

    tris = small_scene("cornellbox1")
    W, H = 64, 36
    d_tris = rt.to_device(tris)
    g = rt.build_geometry(d_tris)
    rg = cedecrt.lookat(*CAM_CB, W, H)
    v1, v2 = rt.buffer(cedecrt.VISIBILITY, W * H), rt.buffer(cedecrt.VISIBILITY, W * H)
    rt.raycast(W, H, g, d_tris, rg, v1)
    rt.launch("raycast", W, H, g, d_tris, rg, v2)
    assert same(v1.to_host(), v2.to_host())
    with pytest.raises(cedecrt.CrtError, match="unknown kernel"):
        rt.launch("no_such_kernel", W)
    with pytest.raises(cedecrt.CrtError, match="too small"):
        rt.raycast(W, H, g, d_tris, rg, rt.buffer(cedecrt.VISIBILITY, 10))


# ------------------------------------------------------------------ full-size properties
def test_full_frame_properties_4k_tiled(rt):
    """BASELINE config 5's size (the blocks_restir stand-in tiled x6 at the real scene's pitch, where the stand-in's copies
    overlap: 9.6 M triangles, 872 k lights; 3840x2160): determinism, pixel classes, and the reference's untouched-output
    rule for sky/emissive pixels"""
    import cedecrt
    import scenes

    tris, cam = scenes.tile_scene(scene("blocks_restir"), 3, 2, 130.0, 82.0), CAM_RESTIR
    W, H = 3840, 2160
    rt.set_math_mode(cedecrt.MATH_LIBDEVICE)
    app = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(accumulate=1, use_temporal_resampling=1,
                                                                use_spatial_resampling=1))
    assert app.lights.n == len(orc.light_indices(tris))
    app.reservoir1.upload(np.full(app.reservoir1.nbytes, 0xAB, np.uint8))  # sentinel: spatial must not touch sky
    app.frame()
    acc1 = app.accumulation.to_host().view(np.float32).reshape(-1, 4)
    vis = app.visibility.to_host()
    out1 = app.output.to_host()
    idx = vis["index"]
    em = (tris["emissive"] > 0).any(1)
    sky = idx < 0
    emi = np.zeros(len(idx), bool)
    emi[~sky] = em[idx[~sky]]
    # the far tiles fill the horizon, so there is less sky than in the untiled frame (14 %)
    assert 0.0 < sky.mean() < 0.1 and 0.01 < emi.mean() < 0.3
    assert (acc1[sky, :3] == 0).all() and (acc1[:, 3] == 1).all()
    assert same(acc1[emi, :3], tris["emissive"][idx[emi]])
    assert np.isfinite(acc1).all() and float(acc1[~sky & ~emi, :3].mean()) > 0
    assert (out1.view(np.uint8).reshape(len(out1), -1)[sky | emi] == 0xAB).all()
    assert (out1["M"][~sky & ~emi] >= 32).all()
    # determinism: a second app from scratch gives the identical frame
    app2 = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(accumulate=1, use_temporal_resampling=1,
                                                                 use_spatial_resampling=1))
    app2.frame()
    assert same(app2.accumulation.to_host(), app.accumulation.to_host())
    assert same(app2.visibility.to_host()["index"], idx)


# ---------------------------------------------------------------------------------------------- fused frame
FUSED_VARIANTS = [
    dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1),
    dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1, spatial_resampling_passes=2),
    dict(accumulate=0, use_temporal_resampling=1, use_spatial_resampling=1, spatial_resampling_passes=1),
    dict(accumulate=1, use_temporal_resampling=0, use_spatial_resampling=1),
    dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=0),
    dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1, use_visibility_reuse=0),
    dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1, use_shadowed_target_function=1),  # per-kernel fallback
    dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1, ris_sample_count=7,
         spatial_resampling_sample_count=3, spatial_resampling_radius=10.0),
]


def diffuse_mask(vis, tris):
    em = (tris["emissive"] > 0).any(1)
    m = vis["index"] >= 0
    m[m] = ~em[vis["index"][m]]
    return m


@pytest.mark.parametrize("variant", range(len(FUSED_VARIANTS)))
def test_fused_frame_bit_exact_vs_oracle(rt, port, variant):
    """crt_restir_di_frame (SoA reservoirs, fused candidate+temporal, conditional visibility-reuse ray, G-buffer,
    tone mapping in the resolve epilogue) against the oracle's kernel-by-kernel chain, exact math mode: every
    buffer the reference's loop leaves behind is reproduced bit for bit."""
    tris = lit_blocks_ao()
    W, H = 160, 90
    kw = FUSED_VARIANTS[variant]
    opt = orc.make_options(**kw)
    rt.set_math_mode(cedecrt.MATH_EXACT)
    port.set_math_mode(1)
    try:
        g = port.geom_build(tris)
        ch = orc.RestirChain(port, W, H, tris, g, *CAM_AO, opt)
        app = cedecrt.RestirDI(rt, W, H, tris, *CAM_AO, cedecrt.Options(**kw), fused=True)
        for _ in range(3):
            ch.step()
            app.frame()
        vis = app.visibility.to_host()
        assert same(vis["index"], ch.vis["index"]) and same(vis["uv"], ch.vis["uv"])
        d = diffuse_mask(ch.vis, tris)
        assert d.sum() > 3000
        if cedecrt.lib().crt_restir_is_fused(app.options):
            temporal = app.export_aos(app.temporal)
        else:
            temporal = app.temporal.to_host()
        assert reservoir_mismatch(ch.temporal, temporal) == 0
        assert reservoir_mismatch(ch.out[d], app.output_reservoirs()[d]) == 0
        acc = app.accumulation.to_host().view(np.float32).reshape(-1, 4)
        assert same(acc, ch.accum)
        assert same(app.pixels.to_host(), port.tone_mapping(ch.accum, W, H))
        port.geom_free(g)
    finally:
        rt.set_math_mode(cedecrt.MATH_LIBDEVICE)
        port.set_math_mode(0)


@pytest.mark.parametrize("name", ["blocks_ao_lit", "blocks_restir"])
def test_fused_equals_per_kernel_path_default_math(rt, name):
    """LIBDEVICE math (uncontracted arithmetic with libdevice's functions, which the launch list and the fused frame share —
    not the context's default, CRT_MATH_REFERENCE, whose contracted kernels only the fused frame has): the fused frame
    and the reference's launch list give identical images"""
    rt.set_math_mode(cedecrt.MATH_LIBDEVICE)
    if name == "blocks_restir":
        tris = scene("blocks_restir")
        W, H, cam, frames = 960, 540, CAM_RESTIR, 3
    else:
        tris, W, H, cam, frames = lit_blocks_ao(), 320, 180, CAM_AO, 4
    kw = dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    a = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(**kw), fused=False)
    b = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(**kw), fused=True)
    for _ in range(frames):
        a.frame()
        b.frame()
    assert same(a.visibility.to_host(), b.visibility.to_host())
    assert same(a.accumulation.to_host(), b.accumulation.to_host())
    assert same(a.pixels.to_host(), b.pixels.to_host())
    va = a.visibility.to_host()
    d = diffuse_mask(va, tris)
    assert reservoir_mismatch(a.temporal.to_host(), b.export_aos(b.temporal)) == 0
    assert reservoir_mismatch(a.output.to_host()[d], b.output_reservoirs()[d]) == 0
    assert float(a.accumulation.to_host().view(np.float32).reshape(-1, 4)[:, :3].sum()) > 0


def test_full_size_band_bit_exact_vs_oracle(rt, port):
    """BASELINE config 5 itself against the oracle: the scene bench.py renders (9.6 M triangles), 3840x2160,
    exact math.  The CPU oracle computes a band of 560 image rows of frames 1 and 2 (every kernel of the loop restricted
    to the band); 3 spatial passes reach 3 x 87 rows, so the 32 central rows of the band see exactly what the full
    frame sees — there the fused frame's primitive ids, uv, temporal reservoirs, final reservoirs, accumulation and
    RGBA8 must equal the oracle's bit for bit."""
    tris, cam = config5()
    W, H, c, half, keep = 3840, 2160, 1080, 280, 16
    kw = dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    rt.set_math_mode(cedecrt.MATH_EXACT)
    port.set_math_mode(1)
    try:
        g = port.geom_build(tris)
        ch = orc.RestirChain(port, W, H, tris, g, *cam, orc.make_options(**kw))
        app = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(**kw), fused=True)
        port.set_range((c - half) * W, (c + half) * W)
        # rows yi in [c - keep, c + keep) of the bottom-up buffers
        rows = slice((H - (c + keep)) * W, (H - (c - keep)) * W)
        for f in range(2):
            ch.step()
            app.frame()
            vis = app.visibility.to_host()[rows]
            assert same(vis["index"], ch.vis["index"][rows]) and same(vis["uv"], ch.vis["uv"][rows]), f
            acc = app.accumulation.to_host().view(np.float32).reshape(-1, 4)[rows]
            assert same(acc, ch.accum[rows]), f
            assert reservoir_mismatch(ch.temporal[rows], app.export_aos(app.temporal)[rows]) == 0, f
            d = diffuse_mask(ch.vis[rows], tris)
            assert d.sum() > 50000
            assert reservoir_mismatch(ch.out[rows][d], app.output_reservoirs()[rows][d]) == 0, f
        pix = app.pixels.to_host().reshape(-1, 4)[rows]
        assert same(pix, port.tone_mapping(ch.accum, W, H).reshape(-1, 4)[rows])
        port.geom_free(g)
    finally:
        port.set_range(0, -1)
        rt.set_math_mode(cedecrt.MATH_LIBDEVICE)
        port.set_math_mode(0)


def test_fused_equals_per_kernel_path_at_full_size(rt):
    """BASELINE config 5 at full size (bench.py's scene, 9.6 M triangles, 3840x2160, temporal + 3 spatial passes +
    visibility reuse): the fused frame bench.py times and the reference's launch list give the same images, bit for
    bit, over three frames — the launch list being the path the small-size tests tie to the oracle kernel by kernel."""
    tris, cam = config5()
    W, H = 3840, 2160
    kw = dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    a = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(**kw), fused=False)
    b = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(**kw), fused=True)
    for f in range(3):
        a.frame()
        b.frame()
        assert same(a.accumulation.to_host(), b.accumulation.to_host()), f
    assert same(a.visibility.to_host(), b.visibility.to_host())
    assert same(a.pixels.to_host(), b.pixels.to_host())
    acc = a.accumulation.to_host().view(np.float32).reshape(-1, 4)
    assert np.isfinite(acc).all() and float(acc[:, :3].sum()) > 0
    d = diffuse_mask(a.visibility.to_host(), tris)
    assert reservoir_mismatch(a.output.to_host()[d], b.output_reservoirs()[d]) == 0


def test_resolve_reuse_of_traced_visibility_changes_no_bit(rt):
    """resolve skips the shadow rays whose answer the reservoir already carries (restir_fast.cuh: kTracedBit); a
    context created with CRT_RESOLVE_REUSE=0 traces every resolve ray like the reference.  Same images, fewer rays."""
    tris = scene("blocks_restir")
    W, H, frames = 960, 540, 4
    kw = dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    os.environ["CRT_RESOLVE_REUSE"] = "0"
    try:
        rt0 = cedecrt.Runtime(0, rt.math_mode)  # the same arithmetic in both contexts (the library's default is REFERENCE)
    finally:
        del os.environ["CRT_RESOLVE_REUSE"]
    try:
        out = []
        for r in (rt, rt0):
            app = cedecrt.RestirDI(r, W, H, tris, *CAM_RESTIR, cedecrt.Options(**kw), fused=True)
            before = r.shadow_rays_traced()
            for _ in range(frames):
                app.frame()
            after = r.shadow_rays_traced()
            out.append((app.accumulation.to_host(), app.pixels.to_host(), app.export_aos(app.temporal),
                        after[0] - before[0], after[1] - before[1], app.visibility.to_host()))
        a, b = out
        assert same(a[0], b[0]) and same(a[1], b[1]) and reservoir_mismatch(a[2], b[2]) == 0
        n_diffuse = int(diffuse_mask(a[5], tris).sum())
        assert b[4] == frames * n_diffuse           # the reference's count: one resolve ray per diffuse pixel
        assert a[3] == b[3] and 0 < a[3] <= frames * n_diffuse
        assert 0.3 * b[4] < a[4] < 0.95 * b[4], (a[4], b[4])
    finally:
        rt0.close()


def test_fused_frame_with_camera_move_and_new_geometry(rt, port):
    """History survives a camera move and a geometry replacement in the reference (it only clears the accumulation on
    a move, 10_restir_di.cpp:257-267, and never rebuilds).  The fused frame's traced-visibility marks must not outlive
    the geometry they were traced against, and a moved camera must not find 'its own' origin in old samples: exact-math
    chain vs oracle across both events."""
    tris_b = lit_blocks_ao()
    tris_a = tris_b.copy()
    # the sequence starts with half of the blocks far away and then they arrive (geometry b): samples that were visible
    # become occluded, which is the case a stale traced mark would get wrong; the lights are the same in both
    tris_a["vertices"][140:1600] += np.float32(500.0)
    W, H = 160, 90
    kw = dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    opt = orc.make_options(**kw)
    rt.set_math_mode(cedecrt.MATH_EXACT)
    port.set_math_mode(1)
    try:
        ga, gb = port.geom_build(tris_a), port.geom_build(tris_b)
        ch = orc.RestirChain(port, W, H, tris_a, ga, *CAM_AO, opt)
        app = cedecrt.RestirDI(rt, W, H, tris_a, *CAM_AO, cedecrt.Options(**kw), fused=True)
        d_tris_b = rt.to_device(tris_b)
        geom_b = rt.build_geometry(d_tris_b)
        cam2 = ((8.5, 7.5, 8.0), (0.0, 0.5, 0.0))
        steps = [("a", CAM_AO), ("a", CAM_AO), ("a", cam2), ("a", cam2), ("b", cam2), ("b", cam2), ("b", CAM_AO)]
        for i, (which, (eye, ctr)) in enumerate(steps):
            ch.eye, ch.rg = np.asarray(eye, np.float32), port.lookat(eye, ctr, W, H)
            app.eye, app.raygen = tuple(float(np.float32(v)) for v in eye), cedecrt.lookat(eye, ctr, W, H)
            if which == "b":
                ch.tris, ch.g = tris_b, gb
                app.triangles, app.geom = d_tris_b, geom_b
            ch.step()
            app.frame()
            acc = app.accumulation.to_host().view(np.float32).reshape(-1, 4)
            assert same(app.visibility.to_host()["index"], ch.vis["index"]), i
            assert same(acc, ch.accum), i
            assert reservoir_mismatch(ch.temporal, app.export_aos(app.temporal)) == 0, i
        port.geom_free(ga)
        port.geom_free(gb)
    finally:
        rt.set_math_mode(cedecrt.MATH_LIBDEVICE)
        port.set_math_mode(0)


def test_reservoir_layout_round_trip(rt):
    n_w, n_h = 64, 16
    n = n_w * n_h
    rng = np.random.default_rng(11)
    a = np.zeros(n, cedecrt.RESERVOIR)
    for f in ("origin_position", "origin_normal", "hit_position", "hit_normal", "radiance"):
        a[f] = rng.standard_normal((n, 3)).astype(np.float32)
    a["visibility"] = rng.integers(0, 2, n)
    a["w_sum"], a["ucw"] = rng.random(n, np.float32), rng.random(n, np.float32)
    a["M"] = rng.integers(0, 2**29 - 1, n)  # 29 bits of M in the record (restir_fast.cuh)
    d_a, d_s, d_b = rt.to_device(a), rt.buffer(cedecrt.RESERVOIR, n), rt.buffer(cedecrt.RESERVOIR, n)
    rt.reservoir_import_aos(n_w, n_h, d_a, d_s)
    rt.reservoir_export_aos(n_w, n_h, d_s, d_b)
    assert reservoir_mismatch(a, d_b.to_host()) == 0


def test_slab_group_on_one_gpu():
    """three row slabs on one GPU, each with its own context and stream, halo rows stored through plain pointers
    (slabs.SlabGroup, what bench.py uses per rank at N > 1): the frame equals the single-slab frame bit for bit"""
    import torch

    import slabs

    tris = scene("blocks_restir")
    W, H = 960, 540
    torch.cuda.set_device(0)
    with torch.cuda.stream(torch.cuda.Stream()):
        part = slabs.SlabGroup(torch, None, 0, 1, tris, CAM_RESTIR, W, H, sub=3)
        part.calibrate(rounds=1, frames=1)
        full = slabs.SlabRenderer(torch, None, 0, 1, tris, CAM_RESTIR, W, H, fused=True)
        for _ in range(4):
            part.frame()
            full.frame()
        torch.cuda.synchronize()
        assert len(set(part.edges)) == 4 and part.edges[0] == 0 and part.edges[-1] == H
        for sl in part.slabs:
            for name, elem in (("t_acc", 16), ("t_pix", 4), ("t_vis", 16)):
                a = sl._rows(getattr(sl, name), elem, sl.y0, sl.y1)
                b = full._rows(getattr(full, name), elem, sl.y0, sl.y1)
                assert torch.equal(a, b), (name, sl.rank)


@pytest.mark.parametrize("mode", ["fused", "fused_nccl", "dropin", "group", "fused_reproject", "dropin_reproject"])
def test_slabs_on_gpus(mode):
    """N row slabs on N GPUs with NCCL halo exchange reproduce the single-GPU frame bit for bit (needs >= 2 GPUs);
    *_reproject: with a moving camera and temporal reprojection, the history rows of every slab gathered by every rank"""
    import subprocess
    import sys

    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 4 if n >= 4 else 2
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                        "--master-addr", "127.0.0.1", "--master-port", str(29700 + os.getpid() % 200),
                        os.path.join(root, "tests", "gpu_slab_worker.py")], env=dict(os.environ, SLAB_MODE=mode),
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "GPU_SLABS_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])
    if mode == "fused":
        assert "p2p True" in r.stdout, r.stdout[-500:]  # the direct-store path really ran
