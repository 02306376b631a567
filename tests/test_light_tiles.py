"""Presampled light tiles (crt_set_light_tiles) without a GPU: the specification's tiles (tests/lights/tile_port.cpp)
against a Python-integer restatement of the draws, their histogram against the source probabilities (chi-square), and
the CUDA path's tile build and candidate bodies (compiled for the host by tests/lights/emu_tiles.cpp) against the
specification bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import orc
from helpers import reservoir_mismatch, same, small_scene
from test_light_sampling import LightPort, light_set

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIGHTS = os.path.join(ROOT, "tests", "lights")
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
F = np.float32
M32, M64 = 0xffffffff, (1 << 64) - 1
CAM_CB = ((0.0, 2.7, 9.0), (0.0, 2.7, 0.0))
CAM_AO = ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class TilePort(LightPort):
    """the light selection's specification with the candidates of generate_candidate drawn from light tiles"""

    def __init__(self, path):
        super().__init__(path)
        self.lib.lt_tile_of.restype = C.c_uint32
        self.tiles = (0, 0)

    def set_light_tiles(self, log2_t, log2_s):
        self.tiles = (log2_t, log2_s)
        self.lib.lt_set_light_tiles(int(log2_t), int(log2_s))

    def tile_slots(self, K, frame):
        out = np.zeros(1 << sum(self.tiles), np.uint32)
        self.lib.lt_tile_slots(C.c_uint32(K), frame, _p(out))
        return out.reshape(1 << self.tiles[0], 1 << self.tiles[1])

    def generate_candidate(self, W, H, frame, g, tris, vis, eye, lights, opt, res=None):
        res = np.zeros(W * H, orc.RESERVOIR) if res is None else res
        eye = np.asarray(eye, np.float32)
        lights = np.ascontiguousarray(lights, np.uint32)
        self.lib.lt_generate_candidate(W, H, frame, g, _p(tris), len(tris), _p(vis), _p(eye), _p(lights), len(lights),
                                       _p(opt), _p(res))
        return res


@pytest.fixture(scope="session")
def tile_port():
    so = os.path.join(LIGHTS, "libtile_port.so")
    subprocess.run([GXX, "-std=c++20", "-O2", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                    "-o", so, os.path.join(LIGHTS, "tile_port.cpp")], check=True)
    p = TilePort(so)
    yield p
    p.set_light_tiles(0, 0)


class EmuTiles(orc.Oracle):
    """tests/emu with generate_candidate drawn from light tiles; the source records and tiles are built the way the
    device builds them (emu_uniform_table / emu_light_table, emu_light_tiles)"""

    def __init__(self, path):
        super().__init__(path)
        self.lib.emu_light_table.restype = C.c_long
        self.lib.emu_light_table.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_long, C.c_void_p]
        self.tiles, self.power = (0, 0), None

    def set_light_tiles(self, log2_t, log2_s):
        self.tiles = (log2_t, log2_s)

    def source(self, tris, lights):
        lights = np.ascontiguousarray(lights, np.uint32)
        if self.power is None:
            out = np.zeros((len(lights), 16), np.float32)
            self.lib.emu_uniform_table(_p(tris), _p(lights), len(lights), _p(out))
            return out
        starts = np.zeros(len(lights) + 1, np.uint32)
        K = self.lib.emu_light_table(_p(tris), _p(lights), len(lights), self.power, None, 0, _p(starts))
        out = np.zeros((K, 16), np.float32)
        assert self.lib.emu_light_table(_p(tris), _p(lights), len(lights), self.power, _p(out), K, _p(starts)) == K
        return out

    def light_tiles(self, src, frame):
        out = np.zeros((1 << sum(self.tiles), 16), np.float32)
        self.lib.emu_light_tiles(_p(src), C.c_uint32(len(src)), frame, self.tiles[0], self.tiles[1], _p(out))
        return out

    def generate_candidate(self, W, H, frame, g, tris, vis, eye, lights, opt, res=None):
        res = np.zeros(W * H, orc.RESERVOIR) if res is None else res
        eye = np.asarray(eye, np.float32)
        tiles = self.light_tiles(self.source(tris, lights), frame)
        self.lib.emu_generate_candidate_tiles(W, H, frame, g, _p(tris), _p(vis), _p(eye), _p(tiles), self.tiles[0],
                                              self.tiles[1], _p(opt), _p(res))
        return res


@pytest.fixture(scope="module")
def emu_tiles():
    so = os.path.join(LIGHTS, "libemu_tiles.so")
    subprocess.run([GXX, "-std=c++17", "-O2", "-fopenmp", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++",
                    "-I" + os.path.join(ROOT, "cedec-2024-rt_b200", "csrc"), "-o", so,
                    os.path.join(LIGHTS, "emu_tiles.cpp")], check=True)
    return EmuTiles(so)


# ---------------------------------------------------------------- the Python restatement
def hash_pcg(v):
    state = (v * 747796405 + 2891336453) & M32
    word = (((state >> ((state >> 28) + 4)) ^ state) * 277803737) & M32
    return (word >> 22) ^ word


def hash_pcg3(x, y, z):
    return hash_pcg((hash_pcg((hash_pcg(x) + y) & M32) + z) & M32)


def pcg_first_f(seed, seq):
    """the first next_f() of Pcg(seed, seq) (common/rng.hpp)"""
    inc = ((seq << 1) | 1) & M64

    def step(s):
        return (s * 6364136223846793005 + inc) & M64

    def out(old):
        xs = (((old >> 18) ^ old) >> 27) & M32
        rot = old >> 59
        return ((xs >> rot) | (xs << ((-rot) & 31))) & M32

    state = step(0)
    state = step((state + seed) & M64)
    u32 = out(state)
    return np.array([(u32 >> 9) | 0x3f800000], np.uint32).view(F)[0] - F(1)


def expected_slots(T, S, K, frame):
    out = np.zeros((T, S), np.uint32)
    for t in range(T):
        for e in range(S):
            s = int(pcg_first_f(hash_pcg3(frame & M32, t, e), 1) * F(K))
            out[t, e] = K - 1 if s == K else s
    return out


@pytest.mark.parametrize("log2_t,log2_s,K,frame", [(0, 4, 37, 1), (3, 5, 1 << 12, 7), (2, 6, 700, -3), (4, 3, 1, 2)])
def test_port_tiles_equal_python_restatement(tile_port, log2_t, log2_s, K, frame):
    tile_port.set_light_tiles(log2_t, log2_s)
    assert same(tile_port.tile_slots(K, frame), expected_slots(1 << log2_t, 1 << log2_s, K, frame))
    want = [hash_pcg3(frame & M32, x >> 3, y >> 2) & ((1 << log2_t) - 1) for x, y in ((0, 0), (13, 6), (100, 41))]
    assert [tile_port.lib.lt_tile_of(x, y, frame) for x, y in ((0, 0), (13, 6), (100, 41))] == want


@pytest.mark.parametrize("source", ["uniform", "power"])
def test_tile_entries_follow_the_source_probabilities(tile_port, source):
    """over many frames the tile entries are drawn by the source's probabilities: chi-square over the lights"""
    n = 40
    tris, lights = light_set(np.random.default_rng(9), n, "dominant" if source == "power" else "random")
    tile_port.set_light_tiles(4, 8)
    if source == "power":
        tile_port.set_light_sampling(1, 10)
        _, starts = tile_port.light_table(tris, lights)
        tile_port.set_light_sampling(0, 0)
        K = 1 << 10
        owner = np.repeat(np.arange(n), np.diff(starts.astype(np.int64)))
        prob = np.diff(starts.astype(np.int64)) / K
    else:
        K, owner, prob = n, np.arange(n), np.full(n, 1.0 / n)
    counts = np.zeros(n, np.int64)
    for frame in range(1, 41):
        counts += np.bincount(owner[tile_port.tile_slots(K, frame).ravel()], minlength=n)
    chi2, pval = stats.chisquare(counts, counts.sum() * prob)
    print("%s: %d draws, chi2 %.1f, p %.3f" % (source, counts.sum(), chi2, pval))
    assert pval > 1e-3


def lit_blocks_ao(n_lights=64):
    tris = small_scene("blocks_ao").copy()
    tris["emissive"][100:100 + n_lights] = np.random.default_rng(3).uniform(0.5, 30.0, (n_lights, 3))
    return tris


SCENES = {"cornellbox1": (lambda: small_scene("cornellbox1"), 64, 36, CAM_CB),
          "lit_blocks_ao": (lit_blocks_ao, 64, 36, CAM_AO)}


@pytest.mark.parametrize("source", ["uniform", "power"])
def test_emu_tile_build_equals_port(tile_port, emu_tiles, source):
    tris = lit_blocks_ao()
    lights = orc.light_indices(tris)
    emu_tiles.power = 10 if source == "power" else None
    try:
        src = emu_tiles.source(tris, lights)
        for tiles, frame in (((3, 5), 1), ((0, 7), 12), ((6, 2), 3)):
            tile_port.set_light_tiles(*tiles)
            emu_tiles.set_light_tiles(*tiles)
            assert same(emu_tiles.light_tiles(src, frame), src[tile_port.tile_slots(len(src), frame).ravel()])
    finally:
        emu_tiles.power = None


def _chain(o, tris, g, opt, W, H, cam, moves=False, frames=3):
    ch = orc.RestirChain(o, W, H, tris, g, *cam, opt, reproject=moves)
    for f in range(frames):
        if moves and f:
            ch.set_camera(tuple(np.asarray(cam[0]) + np.array([0.3, 0.0, -0.2]) * f), cam[1])
        ch.step()
    return ch


def _fused(emu, tris, g, opt, W, H, cam, moves=False, frames=3):
    n = W * H
    vis, prev_vis = np.zeros(n, orc.VISIBILITY), np.zeros(n, orc.VISIBILITY)
    T, A, B = (np.zeros(n * 76, np.uint8) for _ in range(3))
    accum, pixels = np.zeros((n, 4), np.float32), np.zeros(n, np.uint32)
    src = emu.source(tris, orc.light_indices(tris))
    prev_rg, eye = None, cam[0]
    for f in range(frames):
        if moves and f:
            eye = tuple(np.asarray(cam[0]) + np.array([0.3, 0.0, -0.2]) * f)
            accum[:] = 0
        rg = emu.lookat(eye, cam[1], W, H)
        tiles = emu.light_tiles(src, f + 1)
        e = np.asarray(eye, np.float32)
        emu.lib.emu_restir_frame_fast_tiles(W, H, f + 1, g, _p(tris), _p(rg), _p(e), _p(tiles), emu.tiles[0], emu.tiles[1],
                                            _p(opt), _p(vis), _p(T), _p(A), _p(B), _p(accum), _p(pixels),
                                            _p(prev_rg) if (moves and prev_rg is not None) else None, _p(prev_vis))
        prev_rg = rg
        prev_vis[:] = vis
    return accum


@pytest.mark.parametrize("source", ["uniform", "power"])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_device_bodies_equal_the_specification(tile_port, emu_tiles, name, mode, source):
    """px_generate_candidate (the launch list) and px_candidate_temporal (the fused frame, in place and reprojected) over
    LightsTiles against the specification, three frames with temporal and spatial reuse, math mode `mode`"""
    make, W, H, cam = SCENES[name]
    tris = make()
    tiles = (2, 6)
    emu_tiles.power = 10 if source == "power" else None
    for o in (tile_port, emu_tiles):
        o.set_math_mode(mode)
        o.set_light_tiles(*tiles)
    tile_port.set_light_sampling(1 if source == "power" else 0, 10)
    try:
        gp, ge = tile_port.geom_build(tris), emu_tiles.geom_build(tris)
        for kw in (dict(), dict(use_visibility_reuse=0, spatial_resampling_passes=2, ris_sample_count=7)):
            opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1, **kw)
            for moves in (False, True):
                a = _chain(tile_port, tris, gp, opt, W, H, cam, moves)
                b = _chain(emu_tiles, tris, ge, opt, W, H, cam, moves)
                assert reservoir_mismatch(a.out, b.out) == 0 and same(a.accum, b.accum), (kw, moves)
                assert same(_fused(emu_tiles, tris, ge, opt, W, H, cam, moves), a.accum), (kw, moves)
        # tiles change the samples: the image without them differs
        tile_port.set_light_tiles(0, 0)
        assert not same(_chain(tile_port, tris, gp, opt, W, H, cam).accum, a.accum)
        tile_port.geom_free(gp)
        emu_tiles.geom_free(ge)
    finally:
        for o in (tile_port, emu_tiles):
            o.set_math_mode(0)
            o.set_light_tiles(0, 0)
        tile_port.set_light_sampling(0, 0)
        emu_tiles.power = None


def test_tiles_do_not_depend_on_the_row_range(emu_tiles):
    """the candidates of a band of rows, computed alone (orc_set_range), equal the same rows of the whole image"""
    make, W, H, cam = SCENES["lit_blocks_ao"]
    tris = make()
    emu_tiles.set_light_tiles(3, 5)
    g = emu_tiles.geom_build(tris)
    try:
        opt = orc.make_options(accumulate=1)
        rg = emu_tiles.lookat(*cam, W, H)
        vis = emu_tiles.raycast(W, H, g, tris, rg)
        lights = orc.light_indices(tris)
        whole = emu_tiles.generate_candidate(W, H, 2, g, tris, vis, cam[0], lights, opt)
        for t0, t1 in ((0, 13 * W), (13 * W, 29 * W), (29 * W, H * W)):
            emu_tiles.lib.orc_set_range(C.c_long(t0), C.c_long(t1))
            part = emu_tiles.generate_candidate(W, H, 2, g, tris, vis, cam[0], lights, opt)
            emu_tiles.lib.orc_set_range(C.c_long(0), C.c_long(-1))
            idx = np.array([(tid % W) + (H - tid // W - 1) * W for tid in range(t0, t1)])
            assert reservoir_mismatch(part[idx], whole[idx]) == 0
    finally:
        emu_tiles.lib.orc_set_range(C.c_long(0), C.c_long(-1))
        emu_tiles.set_light_tiles(0, 0)
        emu_tiles.geom_free(g)
