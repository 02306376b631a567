"""Reprojection that follows moving geometry (crt_temporal_resampling_reprojected_motion, crt_restir_set_previous_triangles)
without a GPU: the CPU specification (tests/reuse/reuse_port_motion.cpp) against a float64 restatement of p_prev, h, c_h, Z
and ucw on a scene whose triangles are partly translated, partly rotated and partly left alone while the camera moves;
the identity (previous triangles byte-equal to the current ones) against the existing reprojected specification; and the
CUDA path's device bodies (compiled for the host by tests/reuse/emu_reuse_motion.cpp) against the specification bit for
bit, and with floating-point contraction against the existing reprojected bodies under the identity."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import orc
from helpers import reservoir_mismatch, same
from test_reuse_reprojection import MOVES, EmuFusedSurfaces, SurfacesChain, SurfacesEmu, SurfacesPort
from test_reuse_weights import GXX, REUSE, SCENES, VARIANTS, heuristics64, p_hat64, surface64

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def move_triangles(tris, step):
    """The scene after `step` moves: of the non-emissive triangles, index % 3 == 0 are translated, index % 3 == 1 rotated
    about the vertical axis through the scene's centre, index % 3 == 2 left alone (emitters stay: DESIGN.md section 17,
    "Scope").  The moves are small against the scene, so most points stay on screen."""
    out = tris.copy()
    v = tris["vertices"].astype(np.float64)
    lo, hi = v.reshape(-1, 3).min(0), v.reshape(-1, 3).max(0)
    size, centre = float(np.linalg.norm(hi - lo)), (lo + hi) / 2
    idx = np.arange(len(tris))
    still = (tris["emissive"] > 0).any(1)
    tr = (idx % 3 == 0) & ~still
    rot = (idx % 3 == 1) & ~still
    out["vertices"][tr] = (v[tr] + step * size * np.array([0.004, 0.003, -0.002])).astype(F)
    a = 0.01 * step
    c, s = math.cos(a), math.sin(a)
    d = v[rot] - centre
    r = np.stack([c * d[..., 0] + s * d[..., 2], d[..., 1], -s * d[..., 0] + c * d[..., 2]], -1)
    out["vertices"][rot] = (r + centre).astype(F)
    return out


class _Motion:
    """temporal_resampling_motion through the library's rw_temporal_resampling_motion"""

    def temporal_resampling_motion(self, W, H, frame, g, tris, vis, eye, opt, prev_rg, prev_tris, prev_vis, prev, res):
        eye = np.asarray(eye, np.float32)
        self.lib.rw_temporal_resampling_motion(W, H, frame, g, _p(tris), len(tris), _p(vis), _p(eye), _p(opt), _p(prev_rg),
                                               _p(prev_tris), _p(prev_vis), _p(prev), _p(res))
        return res


class MotionPort(_Motion, SurfacesPort):
    pass


class MotionEmu(_Motion, SurfacesEmu):
    pass


def _build(src, so, std, flags, cls, include=False):
    inc = ["-I" + os.path.join(ROOT, "cedec-2024-rt_b200", "csrc")] if include else []
    subprocess.run([GXX, "-std=" + std, "-O2", "-fopenmp", *flags, "-fPIC", "-shared", "-x", "c++", *inc, "-o", so,
                    os.path.join(REUSE, src)], check=True)
    return cls(so)


@pytest.fixture(scope="module")
def spec():
    """tests/reuse/reuse_port_motion.cpp: the specification"""
    return _build("reuse_port_motion.cpp", os.path.join(REUSE, "libreuse_port_motion.so"), "c++20",
                  ["-ffp-contract=off", "-fno-fast-math"], MotionPort)


@pytest.fixture(scope="module")
def emu():
    """tests/reuse/emu_reuse_motion.cpp: the device bodies on the host, as the library's exact build compiles them"""
    return _build("emu_reuse_motion.cpp", os.path.join(REUSE, "libemu_reuse_motion.so"), "c++17", ["-ffp-contract=off"],
                  MotionEmu, include=True)


@pytest.fixture(scope="module")
def emu_contracted():
    """the same with fused multiply-adds allowed (what -fmad=true permits the REFERENCE and FAST builds)"""
    return _build("emu_reuse_motion.cpp", os.path.join(REUSE, "libemu_reuse_motion_contraction.so"), "c++17",
                  ["-ffp-contract=fast", "-mfma"], MotionEmu, include=True)


class MotionChain(SurfacesChain):
    """SurfacesChain whose triangles move: set_triangles() rebuilds the geometry on the new array and keeps the outgoing one;
    the next frame (with a previous camera) calls temporal_resampling_motion with it, as RestirDI.set_triangles does.
    identity=True: the motion call on every frame with a previous camera, with a byte-equal copy of this frame's array.
    static=True: the geometry moves but the temporal step assumes it did not (the previous frame's surfaces call)."""

    def __init__(self, *a, identity=False, static=False, **kw):
        super().__init__(*a, **kw)
        self.prev_tris, self.moved, self.identity, self.static = None, False, identity, static

    def set_triangles(self, tris):
        self.o.geom_free(self.g)
        if not self.moved:
            self.prev_tris = self.tris
        self.tris, self.moved = tris, True
        self.g = self.o.geom_build(tris)

    def temporal_step(self, prev_rg, prev_vis):
        o, W, H, g, t, opt, eye = self.o, self.W, self.H, self.g, self.tris, self.opt, self.eye
        if prev_rg is not None and ((self.moved and not self.static) or self.identity):
            pt = self.prev_tris if self.moved else t.copy()
            self.t_in = self.t_in + (pt,)
            o.temporal_resampling_motion(W, H, self.frame, g, t, self.vis, eye, opt, prev_rg, pt, prev_vis, self.temporal,
                                         self.buf0)
        elif prev_rg is not None:
            o.temporal_resampling_reprojected_surfaces(W, H, self.frame, g, t, self.vis, eye, opt, prev_rg, prev_vis,
                                                       self.temporal, self.buf0)
        else:
            o.temporal_resampling(W, H, self.frame, g, t, self.vis, eye, opt, self.temporal, self.buf0)
        self.moved = False

    def step(self):
        o, W, H = self.o, self.W, self.H
        self.vis, self.prev_vis = self.prev_vis, self.vis
        self.frame += 1
        g, t, opt, eye = self.g, self.tris, self.opt, self.eye
        o.raycast(W, H, g, t, self.rg, self.vis)
        o.generate_candidate(W, H, self.frame, g, t, self.vis, eye, self.lights, opt, self.buf0)
        self.t_in = (self.temporal.copy(), self.buf0.copy(), self.prev_rg, self.prev_vis.copy())
        self.temporal_step(self.prev_rg, self.prev_vis)
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

    def close(self):
        self.o.geom_free(self.g)


class EmuFusedMotion(EmuFusedSurfaces):
    """rw_restir_frame_fast_motion: the fused frame's kernel sequence with crt_restir_set_previous_frame and
    crt_restir_set_previous_triangles on frames after set_triangles; the geometry is rebuilt like MotionChain's"""

    def __init__(self, emu, W, H, tris, eye, center, opt):
        super().__init__(emu, W, H, tris, emu.geom_build(tris), eye, center, opt)
        self.prev_tris, self.moved = None, False

    def set_triangles(self, tris):
        self.emu.geom_free(self.g)
        if not self.moved:
            self.prev_tris = self.tris
        self.tris, self.moved = tris, True
        self.g = self.emu.geom_build(tris)

    def step(self):
        self.vis, self.prev_vis = self.prev_vis, self.vis
        self.frame += 1
        prev = _p(self.prev_rg) if self.prev_rg is not None else None
        pt = _p(self.prev_tris) if self.moved and self.prev_rg is not None else None
        self.moved = False
        self.emu.lib.rw_restir_frame_fast_motion(
            self.W, self.H, self.frame, self.g, _p(self.tris), _p(self.rg), _p(self.eye), _p(self.lights), len(self.lights),
            _p(self.opt), _p(self.vis), _p(self.T), _p(self.A), _p(self.B), _p(self.accum), _p(self.pixels), prev,
            _p(self.prev_vis), pt)
        self.prev_rg = self.rg.copy()

    def close(self):
        self.emu.geom_free(self.g)


def animate(chain, name, scene):
    """two static frames, then twice: the triangles and the camera move, and a frame"""
    for _ in range(2):
        chain.step()
    for k, (eye, center) in enumerate(MOVES[name]):
        chain.set_triangles(move_triangles(scene, k + 1))
        chain.set_camera(eye, center)
        chain.step()
    return chain


def _diffuse(vis, tris):
    d = vis["index"] >= 0
    em = (tris["emissive"] > 0).any(1)
    d[d] = ~em[vis["index"][d]]
    return d


def _moved(tris, prev_tris):
    return (tris["vertices"].view(np.uint32).reshape(len(tris), 9) != prev_tris["vertices"].view(np.uint32).reshape(len(tris), 9)).any(1)


@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_specification_against_float64_restatement(spec, name):
    """The unbiased merge of the last frame, restated in float64 from the specification's own inputs.  p_prev: the point
    on the previous vertices at the record's barycentrics (float32 in the port's order, to 1e-5 of float64), the surface
    point itself on an unmoved triangle; h from orc_reproject_pixel at p_prev; S_h from the previous Visibility at h on the
    previous array's triangle when that triangle moved; c_h = trunc(min(M_h, cap) heuristics(S_q, S_h)), M exactly,
    w_sum and ucw = w_sum / (Z p_hat_q(y)) with Z = c_own [p_hat_q(y) > 0] + c_h [p_hat_h(y) > 0] to a relative 1e-3."""
    make, W, H, cam = SCENES[name]
    scene = make()
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    spec.set_math_mode(1)
    spec.set_reuse_weights(1)
    ch = MotionChain(spec, W, H, scene, spec.geom_build(scene), *cam, opt)
    try:
        animate(ch, name, scene)
    finally:
        spec.set_reuse_weights(0)
        spec.set_math_mode(0)
        ch.close()
    hist, cur, prev_rg, prev_vis, prev_tris = ch.t_in
    tris = ch.tris
    moved = _moved(tris, prev_tris)
    lib = spec.lib
    lib.orc_reproject_pixel.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    eye, eye_prev = ch.eye.astype(np.float64), prev_rg["m_origin"].astype(np.float64)
    cap = 20 * int(opt["ris_sample_count"])
    xy = np.zeros(2, np.int32)
    checked = on_moved = static_h_differs = moved_history = ambiguous = 0
    for q in np.nonzero(_diffuse(ch.vis, tris))[0]:
        v = ch.vis[q]
        t = prev_tris if moved[v["index"]] else tris
        tv = t[v["index"]]["vertices"]
        u, w = F(v["uv"][0]), F(v["uv"][1])
        p32 = np.ascontiguousarray(((F(1) - u - w) * tv[0] + u * tv[1]) + w * tv[2], np.float32)
        p64 = surface64(v, t, eye)[0]
        assert np.abs(p32 - p64).max() <= 1e-5 * max(1.0, np.abs(p64).max())
        s_q = surface64(v, tris, eye)
        own, out = cur[q], ch.t_out[q]
        c_own = int(own["M"])
        prod = None
        if lib.orc_reproject_pixel(prev_rg.ctypes.data, W, H, p32.ctypes.data, xy.ctypes.data):
            h = int(xy[0]) + (H - int(xy[1]) - 1) * W
            if moved[v["index"]]:
                on_moved += 1
                ps = np.ascontiguousarray(surface64(v, tris, eye)[0], np.float32)
                xs = np.zeros(2, np.int32)
                found = lib.orc_reproject_pixel(prev_rg.ctypes.data, W, H, ps.ctypes.data, xs.ctypes.data)
                static_h_differs += not found or int(xs[0]) + (H - int(xs[1]) - 1) * W != h
            hr = hist[h]
            if int(hr["M"]) > 0 and prev_vis[h]["index"] >= 0:
                ht = prev_tris if moved[prev_vis[h]["index"]] else tris
                moved_history += bool(moved[prev_vis[h]["index"]])
                s_h = surface64(prev_vis[h], ht, eye_prev)
                prod = min(int(hr["M"]), cap) * heuristics64(s_q, s_h, eye)
        if prod is None:
            assert int(out["M"]) == c_own and float(out["w_sum"]) == float(own["w_sum"])
            p_q = p_hat64(s_q, out)
            want = float(own["w_sum"]) / (c_own * p_q) if p_q > 0 and c_own > 0 else 0.0
            assert abs(float(out["ucw"]) - want) <= 1e-3 * abs(want), (q, float(out["ucw"]), want)
            checked += 1
            continue
        choices = (round(prod) - 1, round(prod)) if abs(prod - round(prod)) < 1e-4 and round(prod) > 0 else (int(prod),)
        fits = [c for c in choices if c_own + c == int(out["M"])]
        assert fits, (q, prod, c_own, int(out["M"]))
        ambiguous += len(fits) > 1
        c_h = fits[0]
        wsum = float(own["w_sum"]) + p_hat64(s_q, hr) * float(hr["ucw"]) * c_h
        assert abs(float(out["w_sum"]) - wsum) <= 1e-3 * abs(wsum) + 1e-30
        p_q = p_hat64(s_q, out)
        Z = (c_own if p_q > 0 else 0) + (c_h if p_hat64(s_h, out) > 0 else 0)
        want = wsum / (Z * p_q) if p_q > 0 and Z > 0 else 0.0
        assert abs(float(out["ucw"]) - want) <= 1e-3 * abs(want), (q, float(out["ucw"]), want)
        checked += 1
    print("%s: %d merges checked, %d look-ups from moved triangles (%d at another pixel than the static look-up), %d "
          "histories on moved triangles, %d ambiguous" % (name, checked, on_moved, static_h_differs, moved_history, ambiguous))
    assert checked > 500 and on_moved > 0.2 * checked and static_h_differs > 0 and moved_history > 0
    assert ambiguous < 0.01 * checked


@pytest.mark.parametrize("reuse", [0, 1])
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_identity_is_the_reprojected_specification(spec, name, reuse):
    """previous triangles byte-equal to the current ones (a copy) on every frame: the motion specification equals the
    existing reprojected one (k_temporal with a previous camera, k_temporal_unbiased_reprojected) bit for bit"""
    make, W, H, cam = SCENES[name]
    scene = make()
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    spec.set_reuse_weights(reuse)
    try:
        a = MotionChain(spec, W, H, scene, spec.geom_build(scene), *cam, opt, identity=True)
        g = spec.geom_build(scene)
        b = SurfacesChain(spec, W, H, scene, g, *cam, opt)
        for eye, center in [cam] + MOVES[name]:
            for c in (a, b):
                c.set_camera(eye, center)
                c.step()
                c.step()
        assert same(a.accum, b.accum) and reservoir_mismatch(a.temporal, b.temporal) == 0
        assert reservoir_mismatch(a.out, b.out) == 0 and float(a.accum[:, :3].sum()) > 0
        a.close()
        spec.geom_free(g)
    finally:
        spec.set_reuse_weights(0)


@pytest.mark.parametrize("reuse", [0, 1])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("variant", range(len(VARIANTS)))
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_device_bodies_equal_the_specification(spec, emu, name, variant, mode, reuse):
    """px_temporal with MOTION (per-kernel path) and px_candidate_temporal with MOTION (fused frame) against the
    specification while triangles and camera move twice, math mode `mode`, both reuse weights; the fused frame for the
    options it runs (not the shadowed target function).  Ignoring the motion gives other bits."""
    make, W, H, cam = SCENES[name]
    scene = make()
    opt = orc.make_options(**VARIANTS[variant])
    for o in (spec, emu):
        o.set_math_mode(mode)
        o.set_reuse_weights(reuse)
    chains = []
    try:
        a = animate(MotionChain(spec, W, H, scene, spec.geom_build(scene), *cam, opt), name, scene)
        b = animate(MotionChain(emu, W, H, scene, emu.geom_build(scene), *cam, opt), name, scene)
        chains += [a, b]
        assert reservoir_mismatch(a.temporal, b.temporal) == 0 and reservoir_mismatch(a.out, b.out) == 0
        assert same(a.accum, b.accum) and float(a.accum[:, :3].sum()) > 0
        if not opt["use_shadowed_target_function"]:
            f = animate(EmuFusedMotion(emu, W, H, scene, *cam, opt), name, scene)
            chains.append(f)
            d = _diffuse(a.vis, a.tris)
            assert same(f.vis, a.vis) and reservoir_mismatch(f.temporal()[d], a.temporal[d]) == 0
            assert same(f.accum, a.accum)
        # the static assumption (the previous frame's look-up and surfaces on this frame's triangles) is another result
        c = MotionChain(spec, W, H, scene, spec.geom_build(scene), *cam, opt, static=True)
        chains.append(animate(c, name, scene))
        assert reservoir_mismatch(c.temporal, a.temporal) > 0
    finally:
        for o in (spec, emu):
            o.set_math_mode(0)
            o.set_reuse_weights(0)
        for c in chains:
            c.close()


@pytest.mark.parametrize("reuse", [0, 1])
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_identity_of_the_contracted_bodies(emu_contracted, name, reuse):
    """with fused multiply-adds allowed, previous triangles byte-equal to the current ones: the motion bodies equal the
    existing reprojected bodies of the same build bit for bit (p_prev is the surface point itself, not a recomputation;
    S_h is built through the same pointer), per-kernel and fused, in both math modes"""
    make, W, H, cam = SCENES[name]
    scene = make()
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    e = emu_contracted
    e.set_reuse_weights(reuse)
    try:
        for mode in (0, 1):
            e.set_math_mode(mode)
            a = MotionChain(e, W, H, scene, e.geom_build(scene), *cam, opt, identity=True)
            g = e.geom_build(scene)
            b = SurfacesChain(e, W, H, scene, g, *cam, opt)
            fa = EmuFusedMotion(e, W, H, scene, *cam, opt)
            fb = EmuFusedSurfaces(e, W, H, scene, fa.g, *cam, opt)
            for eye, center in [cam] + MOVES[name]:
                for c in (a, b, fa, fb):
                    c.set_camera(eye, center)
                for _ in range(2):
                    for c in (a, b, fb):
                        c.step()
                    fa.moved, fa.prev_tris = True, scene.copy()  # the motion kernel with an unmoved copy
                    fa.step()
            assert same(a.accum, b.accum) and reservoir_mismatch(a.temporal, b.temporal) == 0
            assert same(fa.accum, fb.accum) and reservoir_mismatch(fa.temporal(), fb.temporal()) == 0
            assert float(a.accum[:, :3].sum()) > 0
            a.close()
            e.geom_free(g)
            fa.close()
    finally:
        e.set_math_mode(0)
        e.set_reuse_weights(0)
