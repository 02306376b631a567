"""Pins the oracle (oracle/port, the CPU restatement) before anything trusts it.

1. against the committed golden fixtures (tests/golden/*.npz), which were produced by oracle/_ref —
   the reference's own unmodified .cu files compiled as host C++ (tests/golden/make_golden.py);
2. where oracle/_ref is present (the build container), directly against it on further inputs;
3. against the known-answer values SURVEY.md section 4 extracted from the reference code.

All comparisons are bit-exact.  Mode: math 0 (glibc float functions) + argument order 1 (g++), i.e.
what the reference does as host C++; the canonical GPU order/mode is exercised in test_oracle_modes.
"""
import numpy as np
import pytest

import orc
import helpers
from helpers import golden, reservoir_mismatch, same, small_scene

CAM = ((0.0, 2.7, 9.0), (0.0, 2.7, 0.0))


@pytest.fixture()
def gxx_port(port):
    port.set_math_mode(0)
    port.set_arg_order(1)
    port.set_range(0, -1)
    yield port
    port.set_arg_order(0)


def test_struct_layouts():
    # SURVEY.md section 8a (verified there by compiling the reference headers)
    assert orc.TRIANGLE.itemsize == 60 and orc.VISIBILITY.itemsize == 16 and orc.RESERVOIR.itemsize == 76
    assert orc.OPTIONS.itemsize == 48 and orc.RAYGEN.itemsize == 36
    assert orc.RESERVOIR.fields["visibility"][1] == 60 and orc.RESERVOIR.fields["w_sum"][1] == 64
    assert orc.RESERVOIR.fields["M"][1] == 72
    o = orc.OPTIONS.fields
    assert [o[k][1] for k in ("max_depth", "sky_color", "ris_sample_count", "use_temporal_resampling",
                              "use_spatial_resampling", "spatial_resampling_sample_count",
                              "spatial_resampling_radius", "spatial_resampling_passes",
                              "use_shadowed_target_function", "use_visibility_reuse")] == [4, 8, 20, 28, 29, 32, 36,
                                                                                           40, 44, 45]


def test_scene_goldens_shape():
    cb, ao = small_scene("cornellbox1"), small_scene("blocks_ao")
    assert len(cb) == 36 and len(ao) == 3034  # SURVEY.md section 2.3
    assert len(orc.light_indices(cb)) == 2 and len(orc.light_indices(ao)) == 0
    assert orc.fnv1a64(cb) == "fedadd381237eb3b" and orc.fnv1a64(ao) == "a2d990e76bb6ff22"
    # SURVEY.md section 2.3 quotes FNV-1a-64 values computed from a truncated offset basis (orc.SURVEY_FNV_BASIS):
    # with that start value the loader goldens of the survey are reproduced exactly
    B = orc.SURVEY_FNV_BASIS
    assert orc.fnv1a64(cb, B) == "cc18ef135fe511b9" and orc.fnv1a64(ao, B) == "df1ba0d5b8625ddc"


# SURVEY.md section 4: primary-visibility goldens of the reference's own raycast kernel + core.hpp:91 triangle test on the
# real scenes at the reference cameras, 1920x1080: (sky, emissive, diffuse) pixel counts and FNV-1a-64 (survey basis) of
# the int32 primitive-id image in pixel_idx order.  BASELINE configs 2, 3 and 4/5 (untiled) respectively.
SURVEY_PRIMARY = {
    "blocks_ao": (((8.0, 8.0, 8.0), (0.0, 0.0, 0.0)), (547781, 0, 1525819), "6036eeb91fb634ed", "df1ba0d5b8625ddc"),
    "blocks_pt": (((5.983407, 13.970583, -28.553869), (-5.354514, 4.815835, -2.047728)), (138584, 0, 1935016),
                  "7d6a1cbc62121ca3", "868ff28a3e06c60f"),
    "blocks_restir": (((-0.579885, 22.194597, -6.567105), (5.224952, 20.847435, 1.431192)), (197500, 272518, 1603582),
                      "14de7a5a6a1f96ec", "9d9d4b4ced5814de"),
}


# The same for the stand-ins of the scenes the repository does not hold (helpers.STAND_INS), at the same cameras.  The
# reference has no values for them: these are the port's own output, computed once, so for the port they pin only against
# later changes — and against the reference's own raycast wherever oracle/_ref is built (the test below) — while for the
# CUDA path (test_gpu_configs.py) the port is the independent reference.  blocks_ao is stored whole.
STAND_IN_PRIMARY = {
    "blocks_pt": ((0, 0, 2073600), "101e54971f0cbafd", "eb3b0a7018918863"),
    "blocks_restir": ((292082, 47253, 1734265), "b6cd1761a70aeb50", "69b29d6086b4e5e7"),
}


def primary_goldens(name):
    """(camera, pixel classes, primitive-id hash, scene hash) of the scene helpers.scene(name) returns"""
    cam = SURVEY_PRIMARY[name][0]
    return (cam,) + STAND_IN_PRIMARY[name] if name in STAND_IN_PRIMARY else SURVEY_PRIMARY[name]


def pixel_classes(idx, tris):
    em = (tris["emissive"] > 0).any(1)
    sky = idx < 0
    emi = np.zeros(len(idx), bool)
    emi[~sky] = em[idx[~sky]]
    return int(sky.sum()), int(emi.sum()), int((~sky & ~emi).sum())


@pytest.mark.parametrize("scene", sorted(SURVEY_PRIMARY))
def test_primary_visibility_matches_the_survey_goldens(port, scene):
    """the oracle's raycast (10_restir_di.cu:9-34 restated + the reference triangle test inside oracle/cpu_bvh.h) on the
    scenes of helpers.scene reproduces the goldens bit for bit: scene bytes, pixel classes, primitive-id image — the
    survey's for blocks_ao, STAND_IN_PRIMARY for the stand-ins"""
    cam, classes, prim_hash, scene_hash = primary_goldens(scene)
    tris = helpers.scene(scene)
    assert orc.fnv1a64(tris, orc.SURVEY_FNV_BASIS) == scene_hash
    W, H = 1920, 1080
    g = port.geom_build(tris)
    vis = port.raycast(W, H, g, tris, port.lookat(*cam, W, H))
    port.geom_free(g)
    assert pixel_classes(vis["index"], tris) == classes
    assert orc.fnv1a64(vis["index"], orc.SURVEY_FNV_BASIS) == prim_hash
    if orc.have_reference():  # the reference's own raycast kernel as host C++ gives the same primitive ids
        R = orc.load("reference", 10)
        g = R.geom_build(tris)
        ref = R.raycast(W, H, g, tris, R.lookat(*cam, W, H))
        R.geom_free(g)
        assert same(ref["index"], vis["index"])


def test_restir_chain_matches_reference_golden(gxx_port):
    G = golden("restir_cornell_96x54.npz")
    cb = small_scene("cornellbox1")
    W, H = int(G["W"]), int(G["H"])
    g = gxx_port.geom_build(cb)
    ch = orc.RestirChain(gxx_port, W, H, cb, g, *CAM, G["opt"])
    assert same(ch.rg, G["rg"])
    for _ in range(4):
        ch.step()
    assert same(ch.vis["index"], G["vis"]["index"]) and same(ch.vis["uv"], G["vis"]["uv"])
    assert int((ch.vis["index"] < 0).sum()) == 3554  # SURVEY.md section 4
    for name, buf in (("buf0", ch.buf0), ("buf1", ch.buf1), ("temporal", ch.temporal)):
        assert reservoir_mismatch(buf, G[name]) == 0, name
    assert same(ch.accum, G["accum"])
    assert abs(float(ch.out["M"].mean()) - 115.65567) < 1e-4  # SURVEY.md section 4: mean final M 115.66
    assert same(gxx_port.tone_mapping(ch.accum, W, H), G["pixels"])
    # second option set: shadowed target function, no visibility reuse, 2 passes, 8 candidates
    ch2 = orc.RestirChain(gxx_port, W, H, cb, g, *CAM, G["opt2"])
    ch2.step()
    ch2.step()
    assert reservoir_mismatch(ch2.buf0, G["b_buf0"]) == 0 and reservoir_mismatch(ch2.buf1, G["b_buf1"]) == 0
    assert same(ch2.accum, G["b_accum"])
    gxx_port.geom_free(g)


def test_raycast_blocks_ao_golden(gxx_port):
    G = golden("raycast_blocks_ao_320x180.npz")
    ao = small_scene("blocks_ao")
    W, H = int(G["W"]), int(G["H"])
    g = gxx_port.geom_build(ao)
    rg = gxx_port.lookat((8, 8, 8), (0, 0, 0), W, H)
    assert same(rg, G["rg"])
    vis = gxx_port.raycast(W, H, g, ao, rg)
    assert same(vis["index"], G["vis"]["index"]) and same(vis["uv"], G["vis"]["uv"])
    gxx_port.geom_free(g)


def test_bvh_equals_brute_force(gxx_port):
    """cpu_bvh.h only culls: closest hit == the reference's brute-force loop (04_ao.cu:8-29), incl. the tie rule."""
    import ctypes as C

    ao = small_scene("blocks_ao")
    g = gxx_port.geom_build(ao)
    W, H = 64, 36
    rg = gxx_port.lookat((8, 8, 8), (0, 0, 0), W, H)
    vis = gxx_port.raycast(W, H, g, ao, rg)
    rng = np.random.default_rng(1)
    lib = gxx_port.lib
    lib.orc_closest_hit_brute.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p]
    n_hit = 0
    for _ in range(400):
        o = rng.uniform(-6, 6, 3).astype(np.float32)
        d = rng.normal(size=3).astype(np.float32)
        idx, tuv = gxx_port.closest_hit(g, o, d)
        tuv2 = np.zeros(3, np.float32)
        idx2 = lib.orc_closest_hit_brute(ao.ctypes.data, len(ao), o.ctypes.data, d.ctypes.data, 0.0, 3.402823466e38,
                                         tuv2.ctypes.data)
        assert idx == idx2 and (idx < 0 or same(tuv, tuv2))
        n_hit += idx >= 0
    assert n_hit > 50 and (vis["index"] >= 0).any()
    gxx_port.geom_free(g)


def test_path_tracers_golden(gxx_port):
    G = golden("pt_cornell_96x54.npz")
    cb = small_scene("cornellbox1")
    W, H = 96, 54
    g = gxx_port.geom_build(cb)
    rg = gxx_port.lookat(*CAM, W, H)
    lights = orc.light_indices(cb)
    for ex in (7, 8, 9):
        gxx_port.set_example(ex)
        acc = np.zeros((W * H, 4), np.float32)
        for frame in (1, 2):
            gxx_port.path_trace(W, H, frame, g, cb, lights, rg, G["opt%02d" % ex], acc)
        assert same(acc, G["pt%02d" % ex]), ex
    gxx_port.set_example(9)
    acc = np.zeros((W * H, 4), np.float32)
    gxx_port.path_trace(W, H, 1, g, cb, lights, rg, G["opt09_shadowed"], acc)
    assert same(acc, G["pt09_shadowed"])
    gxx_port.geom_free(g)


def test_ao_goldens(gxx_port):
    G = golden("ao_goldens.npz")
    ao, cb = small_scene("blocks_ao"), small_scene("cornellbox1")
    W, H = int(G["W06"]), int(G["H06"])
    gxx_port.set_example(6)
    g = gxx_port.geom_build(ao)
    assert same(gxx_port.ao(W, H, g, ao, gxx_port.lookat((8, 8, 8), (0, 0, 0), W, H), 64), G["ao06"])
    gxx_port.geom_free(g)
    gxx_port.set_example(4)
    W, H = int(G["W04"]), int(G["H04"])
    assert same(gxx_port.ao(W, H, None, cb, gxx_port.lookat((8, 8, 8), (0, 0, 0), W, H), 64), G["ao04"])
    gxx_port.set_example(9)


def test_rng_known_answers(port):
    """SURVEY.md section 4: values extracted from common/rng.hpp compiled on the host."""
    import ctypes as C

    lib = port.lib
    lib.orc_hash_pcg3.restype = C.c_uint32
    lib.orc_hash_pcg4.restype = C.c_uint32
    assert lib.orc_hash_pcg3(1, 2, 42) == 3300762175
    assert lib.orc_hash_pcg4(0, 0, 1, 0) == 537453139
    # The survey printed `uniform(), uniform(), uniformf()` from one printf argument list, which g++ evaluates
    # right to left: its "1946221658, 2423658439, 0.78417623" are draws 3, 2 and float(draw 1).
    out = np.zeros(3, np.uint32)
    lib.orc_pcg_probe(C.c_uint64(lib.orc_hash_pcg4(3, 5, 1, 0)), C.c_uint64(0), out.ctypes.data)
    assert out.tolist() == [3368011721, 2423658439, 1946221658]
    bits = np.array([(3368011721 >> 9) | 0x3F800000], np.uint32)
    assert abs(float(bits.view(np.float32)[0] - np.float32(1.0)) - 0.78417623) < 1e-8


@pytest.mark.skipif(not orc.have_reference(), reason="oracle/_ref not built (needs /root/reference)")
def test_port_equals_reference_build_directly(gxx_port):
    """Fresh inputs not in the goldens: different resolution, camera and options, blocks_ao with an emissive patch."""
    ao = small_scene("blocks_ao").copy()
    ao["emissive"][100:140] = (5.0, 4.0, 3.0)  # give the light-less scene some emitters
    R = orc.load("reference", 10)
    W, H = 80, 45
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1,
                           spatial_resampling_sample_count=3, spatial_resampling_radius=12.0, ris_sample_count=16)
    outs = []
    for o in (R, gxx_port):
        g = o.geom_build(ao)
        ch = orc.RestirChain(o, W, H, ao, g, (8, 8, 8), (0, 0, 0), opt)
        for _ in range(3):
            ch.step()
        outs.append((ch.vis.copy(), ch.buf0.copy(), ch.buf1.copy(), ch.accum.copy()))
        o.geom_free(g)
    a, b = outs
    assert same(a[0]["index"], b[0]["index"]) and same(a[0]["uv"], b[0]["uv"])
    assert reservoir_mismatch(a[1], b[1]) == 0 and reservoir_mismatch(a[2], b[2]) == 0
    assert same(a[3], b[3])
    assert float(a[3][:, :3].sum()) > 0
