"""Unbiased reuse weights (crt_set_reuse_weights, CRT_REUSE_UNBIASED) without a GPU: the CPU specification
(tests/reuse/reuse_port.cpp) against a float64 restatement of Z and the 1/Z weights, the CUDA path's device bodies
(compiled for the host by tests/reuse/emu_reuse.cpp) against the specification bit for bit, and the identity case in which
the unbiased merge computes the reference's bits."""
import ctypes as C
import itertools
import math
import os
import subprocess

import numpy as np
import pytest

import orc
from helpers import reservoir_mismatch, same, small_scene
from test_light_sampling import LightPort

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REUSE = os.path.join(ROOT, "tests", "reuse")
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
F = np.float32
CAM_CB = ((0.0, 2.7, 9.0), (0.0, 2.7, 0.0))
CAM_AO = ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class _ReuseWeights:
    """temporal_resampling / spatial_resampling through the library's rw_* entry points, which merge with the reference's
    weights (mode 0) or the unbiased ones (mode 1)"""

    def set_reuse_weights(self, mode):
        self.lib.rw_set_reuse_weights(int(mode))

    def temporal_resampling(self, W, H, frame, g, tris, vis, eye, opt, prev, res):
        eye = np.asarray(eye, np.float32)
        self.lib.rw_temporal_resampling(W, H, frame, g, _p(tris), len(tris), _p(vis), _p(eye), _p(opt), _p(prev), _p(res))
        return res

    def spatial_resampling(self, W, H, frame, pas, g, tris, vis, eye, opt, rin, rout):
        eye = np.asarray(eye, np.float32)
        self.lib.rw_spatial_resampling(W, H, frame, pas, g, _p(tris), len(tris), _p(vis), _p(eye), _p(opt), _p(rin), _p(rout))
        return rout


class ReusePort(_ReuseWeights, LightPort):
    """the port of the reference with the light selection of tests/lights/light_port.cpp and the reuse weights of
    tests/reuse/reuse_port.cpp"""


class EmuReuse(_ReuseWeights, orc.Oracle):
    """tests/emu with the device bodies' reuse mode; fused_frame() runs the fused frame's kernel sequence"""


@pytest.fixture(scope="session")
def reuse_port():
    so = os.path.join(REUSE, "libreuse_port.so")
    subprocess.run([GXX, "-std=c++20", "-O2", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                    "-o", so, os.path.join(REUSE, "reuse_port.cpp")], check=True)
    return ReusePort(so)


@pytest.fixture(scope="module")
def emu_reuse():
    so = os.path.join(REUSE, "libemu_reuse.so")
    subprocess.run([GXX, "-std=c++17", "-O2", "-fopenmp", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++",
                    "-I" + os.path.join(ROOT, "cedec-2024-rt_b200", "csrc"), "-o", so,
                    os.path.join(REUSE, "emu_reuse.cpp")], check=True)
    return EmuReuse(so)


def lit_blocks_ao(n_lights=64):
    tris = small_scene("blocks_ao").copy()
    tris["emissive"][100:100 + n_lights] = np.random.default_rng(3).uniform(0.5, 30.0, (n_lights, 3))
    return tris


SCENES = {"cornellbox1": (lambda: small_scene("cornellbox1"), 64, 36, CAM_CB),
          "lit_blocks_ao": (lit_blocks_ao, 64, 36, CAM_AO)}


class ChainWithInputs(orc.RestirChain):
    """orc.RestirChain that keeps, for its last frame, the input of temporal resampling and of every spatial pass"""

    def step(self):
        o, W, H, g, t, opt, eye = self.o, self.W, self.H, self.g, self.tris, self.opt, self.eye
        self.frame += 1
        o.raycast(W, H, g, t, self.rg, self.vis)
        o.generate_candidate(W, H, self.frame, g, t, self.vis, eye, self.lights, opt, self.buf0)
        self.t_in = (self.temporal.copy(), self.buf0.copy())
        o.temporal_resampling(W, H, self.frame, g, t, self.vis, eye, opt, self.temporal, self.buf0)
        self.t_out = self.buf0.copy()
        o.save_temporal_reservoir(W, H, self.buf0, self.temporal)
        self.passes = []
        bi, bo = self.buf0, self.buf1
        for k in range(int(opt["spatial_resampling_passes"])):
            if k != 0:
                bi, bo = bo, bi
            rin = bi.copy()
            o.spatial_resampling(W, H, self.frame, k, g, t, self.vis, eye, opt, bi, bo)
            self.passes.append((rin, bo.copy()))
        self.out = bo
        o.resolve(self.accum, W, H, g, t, self.vis, eye, opt, bo)
        return self.accum


# ---------------------------------------------------------------- the float64 restatement
M64 = (1 << 64) - 1


class Pcg:
    """common/rng.hpp (Python integers)"""

    def __init__(self, seed, seq):
        self.state, self.inc = 0, ((seq << 1) | 1) & M64
        self.next_u32()
        self.state = (self.state + seed) & M64
        self.next_u32()

    def next_u32(self):
        old = self.state
        self.state = (old * 6364136223846793005 + self.inc) & M64
        xs = (((old >> 18) ^ old) >> 27) & 0xffffffff
        rot = old >> 59
        return ((xs >> rot) | (xs << ((-rot) & 31))) & 0xffffffff

    def next_f(self):
        bits = np.array([(self.next_u32() >> 9) | 0x3f800000], np.uint32)
        return bits.view(np.float32)[0] - F(1)


def neighbours(lib, xi, yi, W, H, frame, pas, opt, vis, tris):
    """the pixels the spatial pass visits, in order (the reference's draws in exact math: float32 arithmetic, the
    transcendental functions through double)"""
    lib.orc_hash_pcg4.restype = C.c_uint32
    rng = Pcg(lib.orc_hash_pcg4(xi, yi, frame, 2 + pas), 0)
    R = F(opt["spatial_resampling_radius"])
    out = []
    for _ in range(int(opt["spatial_resampling_sample_count"])):
        rv0, rv1 = rng.next_f(), rng.next_f()
        a = F(-2.0) * F(math.log(float(rv0)))
        radius = np.sqrt(a if a > 0 else F(0))
        phi = F(2.0) * F(3.14159265358979323846) * rv1
        gx, gy = radius * F(math.cos(float(phi))), radius * F(math.sin(float(phi)))
        x, y = int(F(xi) + R / F(1.96) * gx), int(F(yi) + R / F(1.96) * gy)
        if x < 0 or x >= W or y < 0 or y >= H or (x == xi and y == yi):
            continue
        pid = x + (H - y - 1) * W
        if vis[pid]["index"] < 0 or (tris[vis[pid]["index"]]["emissive"] > 0).any():
            continue
        rng.next_f()
        out.append(pid)
    return out


def surface64(vis, tris, eye):
    """make_surface_info (core.hpp:188-207) in float64"""
    t = tris[vis["index"]]["vertices"].astype(np.float64)
    u, v = vis["uv"][0], vis["uv"][1]
    p = (1 - u - v) * t[0] + u * t[1] + v * t[2]
    n = np.cross(t[1] - t[0], t[2] - t[0])
    n /= np.linalg.norm(n)
    if np.dot(eye - p, n) < 0:
        n = -n
    return p, n


def p_hat64(s, y):
    p, n = s
    v = y["hit_position"].astype(np.float64) - p
    d2 = v @ v
    v /= math.sqrt(d2)
    lum = y["radiance"].astype(np.float64) @ np.array([0.1762044, 0.8129847, 0.0108109])
    return abs(v @ n) * abs(-v @ y["hit_normal"].astype(np.float64)) / d2 / math.pi * lum


def heuristics64(s0, s1, eye):
    d0, d1 = np.linalg.norm(s0[0] - eye), np.linalg.norm(s1[0] - eye)
    c = max(float(s0[1] @ s1[1]), 0.0)
    return math.exp(-32.0 * (d1 - d0) ** 2 / d0) * c ** 8


@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_port_against_float64_restatement(reuse_port, name):
    """the unbiased temporal merge and every spatial pass of the third frame, restated in float64 from the port's own
    inputs: M = sum c_j exactly, and w_sum = sum p_hat_q(y_j) ucw_j c_j and ucw = w_sum / (Z p_hat_q(y)) to a relative
    1e-3 (float32 against float64 near grazing angles), with c_j = trunc(M_j * heuristics(S_q, S_j)) on the pixel surfaces.
    A product M_j * heuristics within 1e-4 of an integer k may truncate to k or k - 1 in float32; the choice that gives the
    port's M is taken, and fewer than 1 % of the merges may leave more than one choice open."""
    make, W, H, cam = SCENES[name]
    tris = make()
    eye = np.asarray(cam[0], np.float64)
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    reuse_port.set_math_mode(1)
    reuse_port.set_reuse_weights(1)
    g = reuse_port.geom_build(tris)
    try:
        ch = ChainWithInputs(reuse_port, W, H, tris, g, *cam, opt)
        for _ in range(3):
            ch.step()
    finally:
        reuse_port.set_reuse_weights(0)
        reuse_port.set_math_mode(0)
        reuse_port.geom_free(g)
    diffuse = [i for i in range(W * H) if ch.vis[i]["index"] >= 0 and not (tris[ch.vis[i]["index"]]["emissive"] > 0).any()]
    surf = {i: surface64(ch.vis[i], tris, eye) for i in diffuse}
    checked, ambiguous, z_below_m = 0, 0, 0

    def check(q, own, domains, out):
        """own: the pixel's input reservoir; domains: (reservoir, surface) of the other domains"""
        nonlocal checked, ambiguous, z_below_m
        y = out
        prod = [float(r["M"]) * heuristics64(surf[q], s, eye) for r, s in domains]
        # a product within 1e-4 of an integer k > 0 may truncate to k or k - 1 in float32: the choice that gives M
        choices = [(round(x) - 1, round(x)) if abs(x - round(x)) < 1e-4 and round(x) > 0 else (int(x),) for x in prod]
        fits = [c for c in itertools.product(*choices) if int(own["M"]) + sum(c) == int(out["M"])]
        assert fits, (q, prod, int(own["M"]), int(out["M"]))
        c = fits[0]
        ambiguous += len(fits) > 1
        p_q = p_hat64(surf[q], y)
        w = float(own["w_sum"]) + sum(p_hat64(surf[q], r) * float(r["ucw"]) * cj for (r, _), cj in zip(domains, c))
        assert abs(float(out["w_sum"]) - w) <= 1e-3 * abs(w) + 1e-30
        Z = (int(own["M"]) if p_q > 0 else 0) + sum(cj for (_, s), cj in zip(domains, c) if p_hat64(s, y) > 0)
        z_below_m += Z < int(out["M"])
        want = w / (Z * p_q) if p_q > 0 and Z > 0 else 0.0
        assert abs(float(out["ucw"]) - want) <= 1e-3 * abs(want), (q, float(out["ucw"]), want)
        checked += 1

    hist, cur = ch.t_in
    for q in diffuse:  # temporal: the history's surface is the pixel's own
        h = hist[q].copy()
        h["M"] = min(int(h["M"]), 20 * int(opt["ris_sample_count"]))
        check(q, cur[q], [(h, surf[q])], ch.t_out[q])
    for pas, (rin, rout) in enumerate(ch.passes):
        for q in diffuse:
            yi, xi = H - 1 - q // W, q % W
            nb = neighbours(reuse_port.lib, xi, yi, W, H, 3, pas, opt, ch.vis, tris)
            check(q, rin[q], [(rin[j], surf[j]) for j in nb], rout[q])
    print("%s: %d merges checked, %d with two choices of c_j, Z < M in %d" % (name, checked, ambiguous, z_below_m))
    assert checked > 2000 and ambiguous < 0.01 * checked


def _chain(o, tris, g, opt, W, H, cam, frames=3):
    ch = orc.RestirChain(o, W, H, tris, g, *cam, opt)
    for _ in range(frames):
        ch.step()
    return ch


class EmuFused:
    """rw_restir_frame_fast on planar SoA storage (the kernel sequence of crt_restir_di_frame)"""

    def __init__(self, emu, W, H, tris, g, eye, center, opt):
        self.emu, self.W, self.H, self.tris, self.g, self.opt = emu, W, H, tris, g, opt
        self.eye = np.asarray(eye, np.float32)
        self.rg = emu.lookat(eye, center, W, H)
        self.lights = orc.light_indices(tris)
        n = W * H
        self.vis = np.zeros(n, orc.VISIBILITY)
        self.T, self.A, self.B = (np.zeros(n * 76, np.uint8) for _ in range(3))
        self.accum = np.zeros((n, 4), np.float32)
        self.pixels = np.zeros(n, np.uint32)
        self.frame = 0

    def step(self):
        self.frame += 1
        self.emu.lib.rw_restir_frame_fast(self.W, self.H, self.frame, self.g, _p(self.tris), _p(self.rg), _p(self.eye),
                                          _p(self.lights), len(self.lights), _p(self.opt), _p(self.vis), _p(self.T),
                                          _p(self.A), _p(self.B), _p(self.accum), _p(self.pixels))


VARIANTS = [dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1),
            dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1, use_visibility_reuse=0,
                 spatial_resampling_passes=2, ris_sample_count=7),
            dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1, use_shadowed_target_function=1,
                 ris_sample_count=8)]


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("variant", range(len(VARIANTS)))
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_device_bodies_equal_the_specification(reuse_port, emu_reuse, name, variant, mode):
    """px_temporal / px_spatial (per-kernel path) and px_candidate_temporal / px_spatial_fast (fused frame) in the
    unbiased mode against the CPU specification, three frames with temporal reuse and (by default) 3 spatial passes with
    visibility reuse, math mode `mode`"""
    make, W, H, cam = SCENES[name]
    tris = make()
    opt = orc.make_options(**VARIANTS[variant])
    for o in (reuse_port, emu_reuse):
        o.set_math_mode(mode)
        o.set_reuse_weights(1)
    try:
        gp, ge = reuse_port.geom_build(tris), emu_reuse.geom_build(tris)
        a, b = _chain(reuse_port, tris, gp, opt, W, H, cam), _chain(emu_reuse, tris, ge, opt, W, H, cam)
        assert reservoir_mismatch(a.temporal, b.temporal) == 0 and reservoir_mismatch(a.out, b.out) == 0
        assert same(a.accum, b.accum)
        if not opt["use_shadowed_target_function"]:  # the fused frame's options
            fu = EmuFused(emu_reuse, W, H, tris, ge, *cam, opt)
            for _ in range(3):
                fu.step()
            assert same(fu.accum, a.accum)
        # the unbiased merge is another estimator: the reference's images differ
        reuse_port.set_reuse_weights(0)
        assert not same(_chain(reuse_port, tris, gp, opt, W, H, cam).accum, a.accum)
        reuse_port.geom_free(gp)
        emu_reuse.geom_free(ge)
    finally:
        for o in (reuse_port, emu_reuse):
            o.set_math_mode(0)
            o.set_reuse_weights(0)


def test_reference_mode_of_the_device_bodies_is_the_reference(port, emu_reuse):
    """mode 0 of the templated bodies is the reference's merge: the unchanged port's chain, bit for bit"""
    tris = lit_blocks_ao()
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    gp, ge = port.geom_build(tris), emu_reuse.geom_build(tris)
    a, b = _chain(port, tris, gp, opt, 64, 36, CAM_AO), _chain(emu_reuse, tris, ge, opt, 64, 36, CAM_AO)
    assert same(a.accum, b.accum) and reservoir_mismatch(a.out, b.out) == 0
    fu = EmuFused(emu_reuse, 64, 36, tris, ge, *CAM_AO, opt)
    for _ in range(3):
        fu.step()
    assert same(fu.accum, a.accum)
    port.geom_free(gp)
    emu_reuse.geom_free(ge)


def flat_floor():
    """a floor under one light: every sample's target function is positive at every floor pixel"""
    tris = np.zeros(3, orc.TRIANGLE)
    tris["vertices"][0] = [[-30, 0, -30], [30, 0, -30], [30, 0, 30]]
    tris["vertices"][1] = [[-30, 0, -30], [30, 0, 30], [-30, 0, 30]]
    tris["color"][:2] = 0.7
    tris["vertices"][2] = [[-1, 8, -1], [1, 8, -1], [0, 8, 1.5]]
    tris["emissive"][2] = (40.0, 35.0, 30.0)
    return tris


@pytest.mark.parametrize("mode", [0, 1])
def test_unbiased_equals_reference_on_a_flat_floor(reuse_port, mode):
    """temporal reuse and one spatial pass with one neighbour, no visibility reuse, on a flat floor under one light: every
    sample origin the reference's heuristics read is the pixel surface the unbiased merge reads, and Z = M, so both modes
    compute the same bits.  With more neighbours or passes they part by design: an accepted sample carries its origin."""
    tris = flat_floor()
    W, H, cam = 64, 36, ((0.0, 10.0, 6.0), (0.0, 0.0, 0.0))
    reuse_port.set_math_mode(mode)
    g = reuse_port.geom_build(tris)
    try:
        out = {}
        for k, kw in (("one", dict(spatial_resampling_passes=1, spatial_resampling_sample_count=1)), ("more", {})):
            opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1,
                                   use_visibility_reuse=0, **kw)
            for rw in (0, 1):
                reuse_port.set_reuse_weights(rw)
                ch = _chain(reuse_port, tris, g, opt, W, H, cam, frames=4)
                out[k, rw] = (ch.accum.copy(), ch.out.copy(), ch.temporal.copy())
        ra, ro, rt = out["one", 0]
        ua, uo, ut = out["one", 1]
        assert same(ra, ua) and reservoir_mismatch(ro, uo) == 0 and reservoir_mismatch(rt, ut) == 0
        assert float(ra[:, :3].sum()) > 0
        assert not same(out["more", 0][0], out["more", 1][0])
    finally:
        reuse_port.set_reuse_weights(0)
        reuse_port.set_math_mode(0)
        reuse_port.geom_free(g)
