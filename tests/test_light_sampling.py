"""Power-proportional light selection (crt_set_light_sampling, CRT_LIGHTS_POWER) without a GPU: the port's slot table
against a Python-integer restatement of its formula, the CUDA path's table functions (compiled for the host by tests/emu)
against the port bit for bit, and the identity n = K = 2^k -> power mode == uniform mode on every sampler of the port."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import orc
from helpers import same, small_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32


LIGHTS = os.path.join(ROOT, "tests", "lights")
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


class LightPort(orc.Oracle):
    """the port of the reference with the light selection of tests/lights/light_port.cpp: generate_candidate and
    path_trace (08 / 09) pick lights uniformly or from the power-mode slot table; every other kernel is the port's"""

    def __init__(self, path):
        super().__init__(path)
        L = self.lib
        L.ls_light_table.restype = C.c_long
        L.ls_light_table.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_long, C.c_void_p]
        self.example = 9

    def set_light_sampling(self, mode, log2_slots=0):
        """0 uniform (the reference), 1 in proportion to power from 2^log2_slots slots (0: the default size)"""
        self.lib.ls_set_light_sampling(int(mode), int(log2_slots))

    def light_table(self, tris, lights):
        """(records float32 (K, 16) as the CUDA path's LightRec, starts uint32 (n + 1,)) of the power-mode table, or None
        when 2^log2_slots does not fit the light count"""
        lights = np.ascontiguousarray(lights, np.uint32)
        starts = np.zeros(len(lights) + 1, np.uint32)
        K = self.lib.ls_light_table(_p(tris), _p(lights), len(lights), None, 0, _p(starts))
        if K < 0:
            return None
        out = np.zeros((K, 16), np.float32)
        assert self.lib.ls_light_table(_p(tris), _p(lights), len(lights), _p(out), K, _p(starts)) == K
        return out, starts

    def set_example(self, e):
        self.example = e
        super().set_example(e)

    def generate_candidate(self, W, H, frame, g, tris, vis, eye, lights, opt, res=None):
        res = np.zeros(W * H, orc.RESERVOIR) if res is None else res
        eye = np.asarray(eye, np.float32)
        lights = np.ascontiguousarray(lights, np.uint32)
        self.lib.ls_generate_candidate(W, H, frame, g, _p(tris), len(tris), _p(vis), _p(eye), _p(lights), len(lights),
                                       _p(opt), _p(res))
        return res

    def path_trace(self, W, H, frame, g, tris, lights, rg, opt, accum):
        lights = np.ascontiguousarray(lights, np.uint32)
        self.lib.ls_path_trace_mode(self.example, W, H, frame, g, _p(lights), len(lights), _p(rg), _p(opt), _p(accum))
        return accum


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="session")
def light_port():
    so = os.path.join(LIGHTS, "liblight_port.so")
    subprocess.run([GXX, "-std=c++20", "-O2", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                    "-o", so, os.path.join(LIGHTS, "light_port.cpp")], check=True)
    return LightPort(so)


@pytest.fixture(scope="module")
def emu_lights():
    """the CUDA path's table functions compiled for the host (tests/lights/emu_lights.cpp)"""
    so = os.path.join(LIGHTS, "libemu_lights.so")
    subprocess.run([GXX, "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++",
                    "-I" + os.path.join(ROOT, "cedec-2024-rt_b200", "csrc"), "-o", so,
                    os.path.join(LIGHTS, "emu_lights.cpp")], check=True)
    lib = C.CDLL(so)
    lib.emu_light_table.restype = C.c_long
    lib.emu_light_table.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_long, C.c_void_p]

    def table(tris, lights, log2_slots):
        lights = np.ascontiguousarray(lights, np.uint32)
        starts = np.zeros(len(lights) + 1, np.uint32)
        K = lib.emu_light_table(_p(tris), _p(lights), len(lights), log2_slots, None, 0, _p(starts))
        out = np.zeros((K, 16), np.float32)
        assert lib.emu_light_table(_p(tris), _p(lights), len(lights), log2_slots, _p(out), K, _p(starts)) == K
        return out, starts

    return table


def _cross_len(v):
    a, b = v[:, 1] - v[:, 0], v[:, 2] - v[:, 0]
    c = np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                  a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], 1)
    return c, np.sqrt(c[:, 0] * c[:, 0] + c[:, 1] * c[:, 1] + c[:, 2] * c[:, 2])


def expected_starts(tris, lights, log2_slots):
    """the slot formula restated: float powers (numpy float32, one rounding per operation), integer slot counts"""
    n = len(lights)
    if log2_slots == 0:
        k = min(23, int(np.ceil(np.log2(n))) + 2 if n > 1 else 2)
    else:
        k = log2_slots
    K = 1 << k
    t = tris[lights]
    e = t["emissive"].astype(F)
    lum = e[:, 0] * F(0.1762044) + e[:, 1] * F(0.8129847) + e[:, 2] * F(0.0108109)
    _, ln = _cross_len(t["vertices"].astype(F))
    with np.errstate(invalid="ignore", over="ignore"):
        P = np.where(lum > 0, lum, F(0)) * (F(0.5) * ln)
    P = np.where(P <= np.finfo(F).max, P, F(0)).astype(F)
    pmax = P.max()
    q = [int((P[i] / pmax) * F(2.0 ** 32)) if pmax > 0 else 0 for i in range(n)]
    S, acc = [], 0
    for x in q:
        S.append(acc)
        acc += x
    R = K - n
    starts = [i + (R * S[i] // acc if acc else R * i // n) for i in range(n)] + [K]
    return K, np.array(starts, np.uint32)


def light_set(rng, n, kind):
    """n triangles of random shape whose emission follows `kind`; the light list is every one of them"""
    tris = np.zeros(n, orc.TRIANGLE)
    tris["vertices"] = rng.uniform(-10, 10, (n, 3, 3)).astype(F)
    tris["color"] = 0.5
    if kind == "equal":
        tris["vertices"] = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], F)
        tris["emissive"] = (3.0, 2.0, 1.0)
    elif kind == "dominant":
        tris["emissive"] = rng.uniform(0.01, 0.02, (n, 3))
        tris["emissive"][n // 3] = (1e4, 1e4, 1e4)
    elif kind == "odd":
        tris["emissive"] = rng.uniform(2.0, 40.0, (n, 3))
        k = np.arange(n)
        tris["vertices"][k % 7 == 1] = np.array([[1, 1, 1], [2, 2, 2], [3, 3, 3]], F)  # zero area
        tris["emissive"][k % 7 == 2] = (0.0, 0.0, 0.0)
        tris["emissive"][k % 7 == 3] = (-50.0, 1.0, 1.0)   # negative luminance -> power 0
        tris["emissive"][k % 7 == 4] = (-1.0, 3.0, 0.5)    # a negative channel, positive luminance
        tris["emissive"][k % 7 == 5] = (np.inf, 1.0, 1.0)  # non-finite -> power 0
        tris["emissive"][k % 7 == 6] = (np.nan, 1.0, 1.0)
    else:
        tris["emissive"] = rng.uniform(2.0, 40.0, (n, 3))
    return tris, np.arange(n, dtype=np.uint32)


CASES = [(1, "random", 0), (1, "random", 5), (37, "random", 6), (64, "random", 6), (64, "equal", 0), (1000, "dominant", 0),
         (700, "odd", 0), (700, "odd", 11), (5000, "random", 0), (1000, "dominant", 17)]


def _check_records(tris, lights, K, starts, recs):
    c = np.diff(starts.astype(np.int64))
    owner = np.repeat(np.arange(len(lights)), c)
    t = tris[lights[owner]]
    v = t["vertices"].astype(F)
    cr, ln = _cross_len(v)
    with np.errstate(invalid="ignore", divide="ignore"):
        nrm = cr / ln[:, None]
        sel = c[owner].astype(F) * (F(1) / F(K))
        pdf = sel * F(1) / (F(0.5) * ln)
    want = np.stack([v[:, 0, 0], v[:, 0, 1], v[:, 0, 2], pdf, v[:, 1, 0], v[:, 1, 1], v[:, 1, 2], nrm[:, 0],
                     v[:, 2, 0], v[:, 2, 1], v[:, 2, 2], nrm[:, 1], t["emissive"][:, 0], t["emissive"][:, 1],
                     t["emissive"][:, 2], nrm[:, 2]], 1).astype(F)
    assert same(recs, want)


@pytest.mark.parametrize("n,kind,log2", CASES)
def test_port_slot_table(light_port, n, kind, log2):
    tris, lights = light_set(np.random.default_rng(n + log2), n, kind)
    light_port.set_light_sampling(1, log2)
    try:
        recs, starts = light_port.light_table(tris, lights)
    finally:
        light_port.set_light_sampling(0, 0)
    K, want = expected_starts(tris, lights, log2)
    assert len(recs) == K and same(starts, want)
    c = np.diff(starts.astype(np.int64))
    assert starts[0] == 0 and c.sum() == K and c.min() >= 1
    _check_records(tris, lights, K, starts, recs)
    if kind == "equal":
        assert c.max() - c.min() <= 1
    if kind == "dominant":
        assert c[n // 3] > 0.99 * (K - n)
        if log2 == 17:
            assert c[n // 3] >= 100_000


def test_port_rejects_tables_that_do_not_fit(light_port):
    tris, lights = light_set(np.random.default_rng(1), 100, "random")
    for bad in (6, 24, -1):  # 2^6 < 100 lights; above 2^23; negative
        light_port.set_light_sampling(1, bad)
        assert light_port.light_table(tris, lights) is None
    light_port.set_light_sampling(1, 0)  # no K fits more than 2^23 lights (a list may name a triangle more than once)
    assert light_port.light_table(tris, np.resize(lights, (1 << 23) + 1)) is None
    light_port.set_light_sampling(0, 0)


@pytest.mark.parametrize("n,kind,log2", CASES)
def test_emu_table_equals_port(emu_lights, light_port, n, kind, log2):
    tris, lights = light_set(np.random.default_rng(n + log2), n, kind)
    light_port.set_light_sampling(1, log2)
    try:
        a = light_port.light_table(tris, lights)
    finally:
        light_port.set_light_sampling(0, 0)
    b = emu_lights(tris, lights, log2)
    assert same(a[1], b[1]) and same(a[0], b[0])


def lit_blocks_ao(n_lights=64):
    tris = small_scene("blocks_ao").copy()
    rng = np.random.default_rng(3)
    tris["emissive"][100:100 + n_lights] = rng.uniform(0.5, 30.0, (n_lights, 3))
    return tris


def _restir(port, tris, g, opt, frames=3):
    W, H = 64, 36
    ch = orc.RestirChain(port, W, H, tris, g, (8.0, 8.0, 8.0), (0.0, 0.0, 0.0), opt)
    for _ in range(frames):
        ch.step()
    return ch.accum.copy(), ch.out.copy()


def _paths(port, tris, g, example, opt):
    W, H = 64, 36
    port.set_example(example)
    rg = port.lookat((8.0, 8.0, 8.0), (0.0, 0.0, 0.0), W, H)
    acc = np.zeros((W * H, 4), np.float32)
    port.path_trace(W, H, 1, g, tris, orc.light_indices(tris), rg, opt, acc)
    return acc


@pytest.mark.parametrize("shadowed", [0, 1])
def test_port_power_equals_uniform_when_every_light_owns_one_slot(port, light_port, shadowed):
    """n = K = 2^k: every c_i = 1 and sel_i = 1.0f / (float)n, so power selection computes the bits of the reference's
    uniform selection (the unchanged port) in generate_candidate's 10_restir_di chain, 08_nee and 09_ris"""
    tris = lit_blocks_ao(64)
    assert len(orc.light_indices(tris)) == 64
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1,
                           use_shadowed_target_function=shadowed)
    popt = orc.make_options(accumulate=1, max_depth=3, ris_sample_count=8, use_shadowed_target_function=shadowed)
    out = {}
    for o, mode, log2 in ((port, 0, 0), (light_port, 0, 0), (light_port, 1, 6), (light_port, 1, 8)):
        o.set_math_mode(1)
        g = o.geom_build(tris)
        try:
            if o is light_port:
                o.set_light_sampling(mode, log2)
            out[o.kind if o is port else "ls", mode, log2] = (_restir(o, tris, g, opt), _paths(o, tris, g, 8, popt),
                                                             _paths(o, tris, g, 9, popt))
        finally:
            if o is light_port:
                o.set_light_sampling(0, 0)
            o.set_math_mode(0)
            o.geom_free(g)
    (ra, rr), p8, p9 = out["port", 0, 0]
    for key in (("ls", 0, 0), ("ls", 1, 6)):
        (qa, qr), q8, q9 = out[key]
        assert same(ra, qa) and same(rr, qr) and same(p8, q8) and same(p9, q9), key
    # with K > n the slots go by power: other samples, other images
    (xa, _), x8, x9 = out["ls", 1, 8]
    assert not same(ra, xa) and not same(p8, x8) and not same(p9, x9)
