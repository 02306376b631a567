"""Unbiased reuse weights with a moving camera (crt_temporal_resampling_reprojected_surfaces, crt_restir_set_previous_frame)
without a GPU: the CPU specification (tests/reuse/reuse_port_reprojected.cpp: k_temporal_unbiased_reprojected) against a float64
restatement of c_h, Z and ucw for a camera that moves twice, the CUDA path's device bodies (compiled for the host by
tests/reuse/emu_reuse_reprojected.cpp) against the specification bit for bit, the unmoved-camera identity with the non-reprojected
unbiased merge, and the reference mode of the new bodies against the existing reprojected ones."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import orc
from helpers import reservoir_mismatch, same
from test_reuse_weights import GXX, REUSE, SCENES, VARIANTS, EmuReuse, ReusePort, heuristics64, p_hat64, surface64

F = np.float32
# two camera moves per scene, small enough that most surface points stay on screen.  The Cornell box's second move takes
# the eye past the planes of the right wall (x = 2.76) and the ceiling (y = 5.49), whose far sides it then sees: there the
# previous frame's normal points the other way (its eye was inside), which only the previous eye reproduces.
MOVES = {"cornellbox1": [((1.5, 3.3, 8.4), (0.1, 2.7, 0.0)), ((3.6, 6.0, 8.0), (0.3, 2.6, -2.0))],
         "lit_blocks_ao": [((8.4, 7.8, 8.1), (0.1, 0.0, -0.1)), ((8.9, 7.5, 8.3), (0.2, 0.1, -0.2))]}


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class _Surfaces:
    """temporal_resampling_reprojected_surfaces through the library's rw_temporal_resampling_reprojected"""

    def temporal_resampling_reprojected_surfaces(self, W, H, frame, g, tris, vis, eye, opt, prev_rg, prev_vis, prev, res):
        eye = np.asarray(eye, np.float32)
        self.lib.rw_temporal_resampling_reprojected(W, H, frame, g, _p(tris), len(tris), _p(vis), _p(eye), _p(opt),
                                                    _p(prev_rg), _p(prev_vis), _p(prev), _p(res))
        return res


class SurfacesPort(_Surfaces, ReusePort):
    pass


class SurfacesEmu(_Surfaces, EmuReuse):
    pass


def build_spec():
    """tests/reuse/reuse_port_reprojected.cpp: the specification of the reuse weights with the reprojected temporal merge"""
    so = os.path.join(REUSE, "libreuse_port_reprojected.so")
    subprocess.run([GXX, "-std=c++20", "-O2", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                    "-o", so, os.path.join(REUSE, "reuse_port_reprojected.cpp")], check=True)
    return SurfacesPort(so)


@pytest.fixture(scope="module")
def spec():
    return build_spec()


@pytest.fixture(scope="module")
def emu():
    """tests/reuse/emu_reuse_reprojected.cpp: the device bodies on the host"""
    so = os.path.join(REUSE, "libemu_reuse_reprojected.so")
    subprocess.run([GXX, "-std=c++17", "-O2", "-fopenmp", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++",
                    "-I" + os.path.join(os.path.dirname(REUSE), "..", "cedec-2024-rt_b200", "csrc"), "-o", so,
                    os.path.join(REUSE, "emu_reuse_reprojected.cpp")], check=True)
    return SurfacesEmu(so)


class SurfacesChain(orc.RestirChain):
    """The frame loop with reprojection that keeps two Visibility buffers and passes last frame's on
    (temporal_resampling_reprojected_surfaces from the second frame on); keeps the temporal step's inputs of its last
    frame.  same_surfaces=True: the previous camera and Visibility are this frame's own (the unmoved-camera identity)."""

    def __init__(self, *a, same_surfaces=False, **kw):
        super().__init__(*a, **kw)
        self.prev_vis = np.zeros_like(self.vis)
        self.same_surfaces = same_surfaces

    def step(self):
        o, W, H, g, t, opt, eye = self.o, self.W, self.H, self.g, self.tris, self.opt, self.eye
        self.vis, self.prev_vis = self.prev_vis, self.vis
        self.frame += 1
        o.raycast(W, H, g, t, self.rg, self.vis)
        o.generate_candidate(W, H, self.frame, g, t, self.vis, eye, self.lights, opt, self.buf0)
        prev_rg, prev_vis = (self.rg, self.vis) if self.same_surfaces else (self.prev_rg, self.prev_vis)
        self.t_in = (self.temporal.copy(), self.buf0.copy(), prev_rg, prev_vis.copy())
        if prev_rg is not None:
            o.temporal_resampling_reprojected_surfaces(W, H, self.frame, g, t, self.vis, eye, opt, prev_rg, prev_vis,
                                                       self.temporal, self.buf0)
        else:
            o.temporal_resampling(W, H, self.frame, g, t, self.vis, eye, opt, self.temporal, self.buf0)
        self.t_out = self.buf0.copy()
        self.prev_rg = self.rg
        o.save_temporal_reservoir(W, H, self.buf0, self.temporal)
        bi, bo = self.buf0, self.buf1
        for k in range(int(opt["spatial_resampling_passes"])):
            if k != 0:
                bi, bo = bo, bi
            o.spatial_resampling(W, H, self.frame, k, g, t, self.vis, eye, opt, bi, bo)
        self.out = bo
        o.resolve(self.accum, W, H, g, t, self.vis, eye, opt, bo)
        return self.accum


def moving(chain, name):
    """two static frames, then a move and a frame, twice"""
    for _ in range(2):
        chain.step()
    for eye, center in MOVES[name]:
        chain.set_camera(eye, center)
        chain.step()
    return chain


class EmuFusedSurfaces:
    """rw_restir_frame_fast_reprojected: the fused frame's kernel sequence with crt_restir_set_previous_frame (two
    Visibility buffers, alternated; the history read from a snapshot of `temporal`) or, reproject=False, without"""

    def __init__(self, emu, W, H, tris, g, eye, center, opt, reproject=True):
        self.emu, self.W, self.H, self.tris, self.g, self.opt, self.reproject = emu, W, H, tris, g, opt, reproject
        self.eye = np.asarray(eye, np.float32)
        self.rg = emu.lookat(eye, center, W, H)
        self.prev_rg = None
        self.lights = orc.light_indices(tris)
        n = W * H
        self.vis, self.prev_vis = np.zeros(n, orc.VISIBILITY), np.zeros(n, orc.VISIBILITY)
        self.T, self.A, self.B = (np.zeros(n * 76, np.uint8) for _ in range(3))
        self.accum = np.zeros((n, 4), np.float32)
        self.pixels = np.zeros(n, np.uint32)
        self.frame = 0

    def set_camera(self, eye, center):
        self.eye = np.asarray(eye, np.float32)
        self.rg = self.emu.lookat(eye, center, self.W, self.H)
        self.accum[:] = 0

    def step(self):
        self.vis, self.prev_vis = self.prev_vis, self.vis
        self.frame += 1
        prev = _p(self.prev_rg) if self.reproject and self.prev_rg is not None else None
        self.emu.lib.rw_restir_frame_fast_reprojected(
            self.W, self.H, self.frame, self.g, _p(self.tris), _p(self.rg), _p(self.eye), _p(self.lights), len(self.lights),
            _p(self.opt), _p(self.vis), _p(self.T), _p(self.A), _p(self.B), _p(self.accum), _p(self.pixels), prev,
            _p(self.prev_vis))
        self.prev_rg = self.rg.copy()

    def temporal(self):
        out = np.zeros(self.W * self.H, orc.RESERVOIR)
        self.emu.lib.emu_soa_to_aos(_p(self.T), _p(out), C.c_long(len(out)))
        return out


def _diffuse(vis, tris):
    d = vis["index"] >= 0
    em = (tris["emissive"] > 0).any(1)
    d[d] = ~em[vis["index"][d]]
    return d


def _surface_point32(v, tris):
    """bary_point of make_surface_info (core.hpp:188-207) in float32, the operations in the port's order"""
    t = tris[v["index"]]["vertices"]
    u, w = F(v["uv"][0]), F(v["uv"][1])
    return ((F(1) - u - w) * t[0] + u * t[1]) + w * t[2]


@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_specification_against_float64_restatement(spec, name):
    """the reprojected unbiased temporal merge of the last frame of a camera that moved twice, restated in float64 from
    the specification's own inputs: h from orc_reproject_pixel, S_h from the previous Visibility at h with the previous
    eye, c_h = trunc(min(M_h, cap) * heuristics(S_q, S_h)), M = c_own + c_h exactly, w_sum and ucw = w_sum / (Z p_hat_q(y))
    with Z = c_own [p_hat_q(y) > 0] + c_h [p_hat_h(y) > 0] to a relative 1e-3.  A product within 1e-4 of an integer k may
    truncate to k or k - 1 in float32: the choice that gives the specification's M is taken (fewer than 1 % of merges)."""
    make, W, H, cam = SCENES[name]
    tris = make()
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    spec.set_math_mode(1)
    spec.set_reuse_weights(1)
    g = spec.geom_build(tris)
    try:
        ch = moving(SurfacesChain(spec, W, H, tris, g, *cam, opt), name)
    finally:
        spec.set_reuse_weights(0)
        spec.set_math_mode(0)
        spec.geom_free(g)
    hist, cur, prev_rg, prev_vis = ch.t_in
    lib = spec.lib
    lib.orc_reproject_pixel.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    eye, eye_prev = ch.eye.astype(np.float64), prev_rg["m_origin"].astype(np.float64)
    cap = 20 * int(opt["ris_sample_count"])
    xy = np.zeros(2, np.int32)
    checked = ambiguous = moved = other_surface = 0
    for q in np.nonzero(_diffuse(ch.vis, tris))[0]:
        p32 = np.ascontiguousarray(_surface_point32(ch.vis[q], tris), np.float32)
        s_q = surface64(ch.vis[q], tris, eye)
        own, out = cur[q], ch.t_out[q]
        y = out
        c_own = int(own["M"])
        prod = None
        if lib.orc_reproject_pixel(prev_rg.ctypes.data, W, H, p32.ctypes.data, xy.ctypes.data):
            h = int(xy[0]) + (H - int(xy[1]) - 1) * W
            moved += h != q
            hr = hist[h]
            if int(hr["M"]) > 0 and prev_vis[h]["index"] >= 0:
                s_h = surface64(prev_vis[h], tris, eye_prev)
                other_surface += prev_vis[h]["index"] != ch.vis[q]["index"]
                prod = min(int(hr["M"]), cap) * heuristics64(s_q, s_h, eye)
        if prod is None:  # no history domain: the merge keeps this frame's reservoir up to the weight-0 merge
            assert int(out["M"]) == c_own and float(out["w_sum"]) == float(own["w_sum"])
            p_q = p_hat64(s_q, y)
            want = float(own["w_sum"]) / (c_own * p_q) if p_q > 0 and c_own > 0 else 0.0
            assert abs(float(out["ucw"]) - want) <= 1e-3 * abs(want), (q, float(out["ucw"]), want)
            checked += 1
            continue
        choices = (round(prod) - 1, round(prod)) if abs(prod - round(prod)) < 1e-4 and round(prod) > 0 else (int(prod),)
        fits = [c for c in choices if c_own + c == int(out["M"])]
        assert fits, (q, prod, c_own, int(out["M"]))
        ambiguous += len(fits) > 1
        c_h = fits[0]
        w = float(own["w_sum"]) + p_hat64(s_q, hr) * float(hr["ucw"]) * c_h
        assert abs(float(out["w_sum"]) - w) <= 1e-3 * abs(w) + 1e-30
        p_q = p_hat64(s_q, y)
        Z = (c_own if p_q > 0 else 0) + (c_h if p_hat64(s_h, y) > 0 else 0)
        want = w / (Z * p_q) if p_q > 0 and Z > 0 else 0.0
        assert abs(float(out["ucw"]) - want) <= 1e-3 * abs(want), (q, float(out["ucw"]), want)
        checked += 1
    print("%s: %d merges checked, %d look-ups at another pixel, %d on another triangle, %d ambiguous"
          % (name, checked, moved, other_surface, ambiguous))
    assert checked > 500 and moved > 0.5 * checked and other_surface > 0 and ambiguous < 0.01 * checked


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("variant", range(len(VARIANTS)))
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_device_bodies_equal_the_specification(spec, emu, name, variant, mode):
    """px_temporal with a previous camera and the previous Visibility (per-kernel path) and px_candidate_temporal with
    REPROJ (fused frame, crt_restir_set_previous_frame) in the unbiased mode against the specification, camera moving
    twice, math mode `mode`; the fused frame for the options it runs (not the shadowed target function)"""
    make, W, H, cam = SCENES[name]
    tris = make()
    opt = orc.make_options(**VARIANTS[variant])
    for o in (spec, emu):
        o.set_math_mode(mode)
        o.set_reuse_weights(1)
    gp, ge = spec.geom_build(tris), emu.geom_build(tris)
    try:
        a = moving(SurfacesChain(spec, W, H, tris, gp, *cam, opt), name)
        b = moving(SurfacesChain(emu, W, H, tris, ge, *cam, opt), name)
        assert reservoir_mismatch(a.temporal, b.temporal) == 0 and reservoir_mismatch(a.out, b.out) == 0
        assert same(a.accum, b.accum) and float(a.accum[:, :3].sum()) > 0
        if not opt["use_shadowed_target_function"]:
            f = moving(EmuFusedSurfaces(emu, W, H, tris, ge, *cam, opt), name)
            d = _diffuse(a.vis, tris)
            assert same(f.vis, a.vis) and reservoir_mismatch(f.temporal()[d], a.temporal[d]) == 0
            assert same(f.accum, a.accum)
        # the reference's reprojected chain is another estimator
        spec.set_reuse_weights(0)
        assert not same(moving(SurfacesChain(spec, W, H, tris, gp, *cam, opt), name).accum, a.accum)
    finally:
        for o in (spec, emu):
            o.set_math_mode(0)
            o.set_reuse_weights(0)
        spec.geom_free(gp)
        emu.geom_free(ge)


@pytest.mark.parametrize("variant", range(len(VARIANTS)))
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_unmoved_camera_is_the_unreprojected_unbiased_merge(spec, emu, name, variant):
    """previous camera = this camera and previous Visibility = this frame's: the look-up is the pixel itself and S_h = S_q,
    so the new merge computes section 15's non-reprojected unbiased merge bit for bit (specification and device bodies)"""
    make, W, H, cam = SCENES[name]
    tris = make()
    opt = orc.make_options(**VARIANTS[variant])
    for o in (spec, emu):
        o.set_reuse_weights(1)
    try:
        for o in (spec, emu):
            g = o.geom_build(tris)
            a = SurfacesChain(o, W, H, tris, g, *cam, opt, same_surfaces=True)
            b = orc.RestirChain(o, W, H, tris, g, *cam, opt)
            for _ in range(4):
                a.step()
                b.step()
            assert same(a.accum, b.accum) and reservoir_mismatch(a.temporal, b.temporal) == 0
            assert reservoir_mismatch(a.out, b.out) == 0 and float(a.accum[:, :3].sum()) > 0
            o.geom_free(g)
    finally:
        for o in (spec, emu):
            o.set_reuse_weights(0)


@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_reference_mode_of_the_new_bodies_is_the_reprojected_reference(port, spec, emu, name):
    """under the reference's weights the previous Visibility is not read: the new per-kernel and fused bodies equal the
    existing reprojected ones (the port's k_temporal with a previous camera, emu_restir_frame_fast_reprojected)"""
    make, W, H, cam = SCENES[name]
    tris = make()
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    gp, gs, ge = port.geom_build(tris), spec.geom_build(tris), emu.geom_build(tris)
    ref = moving(orc.RestirChain(port, W, H, tris, gp, *cam, opt, reproject=True), name)
    for o, g in ((spec, gs), (emu, ge)):
        ch = moving(SurfacesChain(o, W, H, tris, g, *cam, opt), name)
        assert same(ch.accum, ref.accum) and reservoir_mismatch(ch.temporal, ref.temporal) == 0
        assert reservoir_mismatch(ch.out, ref.out) == 0
    f = moving(EmuFusedSurfaces(emu, W, H, tris, ge, *cam, opt), name)
    assert same(f.accum, ref.accum)
    port.geom_free(gp)
    spec.geom_free(gs)
    emu.geom_free(ge)
