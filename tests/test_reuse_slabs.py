"""Halo surfaces (crt_restir_set_halo_surfaces) without a GPU: the body that writes the G-buffer records of rows outside a
context's range (csrc/restir_fast.cuh: px_halo_surface, compiled for the host by tests/reuse/emu_halo_surfaces.cpp) against
the records the candidate kernel's body (px_candidate_temporal) stores for the same pixels on the context that owns them —
bit for bit, with and without floating-point contraction, over a camera that moves twice.  Also the host-side reach of
the halo bands (slabs.halo_rows, the same formula as csrc: halo_rows_for)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import orc
from test_reuse_reprojection import MOVES
from test_reuse_weights import GXX, REUSE, SCENES, EmuReuse

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module", params=["no_contraction", "contraction"])
def emu(request):
    """the device bodies on the host, with -ffp-contract=off (the library's exact build) or with fused multiply-adds allowed
    (what -fmad=true permits the REFERENCE and FAST builds): both bodies are compiled the same way in each"""
    contract = request.param == "contraction"
    so = os.path.join(REUSE, "libemu_halo_surfaces_%s.so" % request.param)
    flags = ["-ffp-contract=fast", "-mfma"] if contract else ["-ffp-contract=off"]
    subprocess.run([GXX, "-std=c++17", "-O2", "-fopenmp", *flags, "-fPIC", "-shared", "-x", "c++",
                    "-I" + os.path.join(ROOT, "cedec-2024-rt_b200", "csrc"), "-o", so,
                    os.path.join(REUSE, "emu_halo_surfaces.cpp")], check=True)
    return EmuReuse(so)


def _diffuse(vis, tris):
    d = vis["index"] >= 0
    em = (tris["emissive"] > 0).any(1)
    d[d] = ~em[vis["index"][d]]
    return d


@pytest.mark.parametrize("reuse", [0, 1])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_halo_records_equal_the_owners_records(emu, name, mode, reuse):
    """for every frame of a camera that moves twice: the owners' G-buffer (px_candidate_temporal over the whole image)
    against px_halo_surface over two bands of rows, written into buffers poisoned beforehand.  Diffuse pixels: the same 24
    bytes.  Sky and emissive pixels: no record (still poisoned).  The class plane: never written."""
    make, W, H, cam = SCENES[name]
    tris = make()
    lib = emu.lib
    emu.set_math_mode(mode)
    emu.set_reuse_weights(reuse)
    g = emu.geom_build(tris)
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    lights = orc.light_indices(tris)
    n = W * H
    temporal = np.zeros(n * 76, np.uint8)
    bands = [(0, 11), (23, H)]  # edges on no multiple of 8; rows 11..22 are the "own" rows left out
    checked = flipped = 0
    try:
        cams = [cam, cam] + MOVES[name]
        prev_eye = None
        for f, (e, ctr) in enumerate(cams, 1):
            eye = np.asarray(e, np.float32)
            rg = emu.lookat(e, ctr, W, H)
            vis = np.zeros(n, orc.VISIBILITY)
            emu.raycast(W, H, g, tris, rg, vis)
            own = (np.zeros(n * 16, np.uint8), np.zeros(n * 8, np.uint8), np.zeros(n, np.uint8))
            lib.hs_candidate_gbuf(W, H, f, g, _p(tris), _p(vis), _p(eye), _p(lights), len(lights), _p(opt), _p(temporal),
                                  *(_p(a) for a in own))
            halo = (np.full(n * 16, 0xAB, np.uint8), np.full(n * 8, 0xAB, np.uint8), np.full(n, 0xAB, np.uint8))
            for y0, y1 in bands:
                lib.hs_halo_gbuf(W, H, y0, y1, _p(tris), _p(vis), _p(eye), *(_p(a) for a in halo))
            yi = (H - 1) - np.arange(n) // W  # pixel_idx = xi + (H - yi - 1) * W
            in_band = np.zeros(n, bool)
            for y0, y1 in bands:
                in_band |= (yi >= y0) & (yi < y1)
            d = _diffuse(vis, tris)
            g0o, g1o = own[0].reshape(n, 16), own[1].reshape(n, 8)
            g0h, g1h = halo[0].reshape(n, 16), halo[1].reshape(n, 8)
            assert (g0h[d & in_band] == g0o[d & in_band]).all() and (g1h[d & in_band] == g1o[d & in_band]).all(), f
            assert (g0h[~(d & in_band)] == 0xAB).all() and (g1h[~(d & in_band)] == 0xAB).all(), f
            assert (halo[2] == 0xAB).all()
            checked += int((d & in_band).sum())
            if prev_eye is not None and name == "cornellbox1" and f == len(cams):
                # the eye is part of the record: the previous eye gives another normal where the camera crossed a wall's plane
                stale = (np.full(n * 16, 0xAB, np.uint8), np.full(n * 8, 0xAB, np.uint8), np.full(n, 0xAB, np.uint8))
                for y0, y1 in bands:
                    lib.hs_halo_gbuf(W, H, y0, y1, _p(tris), _p(vis), _p(prev_eye), *(_p(a) for a in stale))
                flipped = int((stale[0].reshape(n, 16)[d & in_band] != g0o[d & in_band]).any(1).sum() +
                              (stale[1].reshape(n, 8)[d & in_band] != g1o[d & in_band]).any(1).sum())
                assert flipped > 0
            prev_eye = eye
    finally:
        emu.set_math_mode(0)
        emu.set_reuse_weights(0)
        emu.geom_free(g)
    assert checked > 0.25 * len(cams) * sum(b - a for a, b in bands) * W


def test_halo_reach():
    """the rows a spatial pass can reach beyond its own (include/cedecrt.h: crt_restir_set_halo_surfaces): 87 at the
    reference's radius 30 (slabs.HALO, the direct-store links' band), more at a larger radius"""
    import slabs

    assert slabs.halo_rows(30) == slabs.HALO == 87
    assert slabs.halo_rows(45) > 87 and slabs.halo_rows(10) < 87
