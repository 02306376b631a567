"""Presampled light tiles on the GPU (crt_set_light_tiles): the device tiles against the specification's draws byte for
byte, the launch list, the fused frame and its per-kernel path bit for bit against the specification in EXACT mode, row
ranges and slabs against one context, switching off, the refusals, and unbiasedness against selection without tiles."""
import numpy as np
import pytest

import orc
from helpers import DeviceAsOracle, same, scene, small_scene
from test_gpu_light_sampling import lit_blocks_ao, one_bright_many_dim, CAM_FLOOR
from test_light_tiles import tile_port  # noqa: F401  (the fixture)

pytestmark = pytest.mark.gpu
CAM_AO = ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0))
CAM_CB = ((0.0, 2.7, 9.0), (0.0, 2.7, 0.0))
CAM_RESTIR = ((0.0, 22.0, 0.0), (30.0, 18.0, 30.0))
EINVAL = 3  # include/cedecrt.h: CRT_EINVAL


@pytest.fixture(scope="module")
def rt():
    import cedecrt

    r = cedecrt.Runtime(0, cedecrt.MATH_EXACT)
    yield r
    r.close()


@pytest.fixture()
def c(rt):
    import cedecrt

    rt.set_math_mode(cedecrt.MATH_EXACT)
    yield cedecrt
    rt.set_light_tiles(0, 0)
    rt.set_light_sampling(cedecrt.LIGHTS_UNIFORM)
    rt.set_reuse_weights(cedecrt.REUSE_REFERENCE)


@pytest.fixture()
def spec(tile_port):  # noqa: F811
    tile_port.set_math_mode(1)
    yield tile_port
    tile_port.set_light_tiles(0, 0)
    tile_port.set_light_sampling(0, 0)
    tile_port.set_math_mode(0)


@pytest.mark.parametrize("source", ["uniform", "power"])
def test_device_tiles_equal_the_specification(rt, c, spec, source):
    tris = scene("blocks_restir") if source == "power" else lit_blocks_ao()
    lights = orc.light_indices(tris)
    d_t, d_l = rt.to_device(tris), rt.to_device(lights)
    g = rt.build_geometry(d_t)
    rt.set_light_sampling(c.LIGHTS_POWER if source == "power" else c.LIGHTS_UNIFORM)
    try:
        src = rt.light_sampling_table(g, d_l)
        for tiles, frame in (((7, 10), 1), ((3, 5), 2), ((0, 12), 17), ((10, 0), 3)):
            rt.set_light_tiles(*tiles)
            spec.set_light_tiles(*tiles)
            got = rt.light_tiles(g, d_l, frame)
            want = src[spec.tile_slots(len(src), frame)]
            assert got.shape == want.shape and same(got, want), (tiles, frame)
    finally:
        g.destroy()


def _chain(o, tris, g, opt, W, H, cam, moves=False, frames=3):
    ch = orc.RestirChain(o, W, H, tris, g, *cam, opt, reproject=moves)
    for f in range(frames):
        if moves and f:
            ch.set_camera(tuple(np.asarray(cam[0]) + np.array([0.3, 0.0, -0.2]) * f), cam[1])
        ch.step()
    return ch


def _fused(rt, c, tris, opt, W, H, cam, moves=False, frames=3, overlap=False):
    app = c.RestirDI(rt, W, H, tris, *cam, c.Options.from_numpy(opt), fused=True, reproject=moves)
    if overlap:
        rt.set_frame_overlap(1)
        app.prefetch = True
    try:
        for f in range(frames):
            if moves and f:
                app.set_camera(tuple(np.asarray(cam[0]) + np.array([0.3, 0.0, -0.2]) * f), cam[1])
            app.frame()
        rt.sync()
        acc = app.accumulation.to_host().view(np.float32).reshape(-1, 4).copy()
    finally:
        if overlap:
            rt.set_frame_overlap(0)
    app.geom.destroy()
    return acc


class Launched(DeviceAsOracle):
    """DeviceAsOracle whose generate_candidate goes through crt_launch by name"""

    def generate_candidate(self, W, H, frame, g, tris, vis, eye, lights, opt, res=None):
        bufs = [self.rt.to_device(a) for a in (tris, vis, np.ascontiguousarray(lights, np.uint32))]
        out = self.rt.to_device(res if res is not None else np.zeros(W * H, orc.RESERVOIR))
        e = self.c.Float3(*[float(np.float32(v)) for v in eye])
        self.rt.launch("generate_candidate", W, H, frame, g, bufs[0], bufs[1], e, bufs[2], self._opt(opt), out)
        r = out.to_host().view(orc.RESERVOIR)
        if res is not None:
            res[:] = r
            return res
        return r


@pytest.mark.parametrize("source", ["uniform", "power"])
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_exact_tiles_equal_the_specification(rt, c, spec, name, source):
    """the launch list (typed call and crt_launch), the fused frame (in place, reprojected, with frame overlap and the
    primary-ray prefetch) and its per-kernel path (shadowed target function), 3 frames, bit for bit"""
    tris = lit_blocks_ao() if name == "lit_blocks_ao" else small_scene("cornellbox1")
    cam = CAM_AO if name == "lit_blocks_ao" else CAM_CB
    W, H = 160, 90
    power = source == "power"
    spec.set_light_sampling(1 if power else 0, 0)
    rt.set_light_sampling(c.LIGHTS_POWER if power else c.LIGHTS_UNIFORM)
    spec.set_light_tiles(3, 7)
    rt.set_light_tiles(3, 7)
    gp = spec.geom_build(tris)
    base = dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    for kw in (base, dict(base, use_visibility_reuse=0), dict(base, use_shadowed_target_function=1)):
        opt = orc.make_options(**kw)
        a = _chain(spec, tris, gp, opt, W, H, cam)
        for dev in (DeviceAsOracle(rt), Launched(rt)):
            b = _chain(dev, tris, dev.geom_build(tris), opt, W, H, cam)
            assert same(a.accum, b.accum) and same(a.out, b.out), (kw, type(dev).__name__)
        assert same(_fused(rt, c, tris, opt, W, H, cam), a.accum), kw
    opt = orc.make_options(**base)
    a = _chain(spec, tris, gp, opt, W, H, cam, moves=True)
    dev = DeviceAsOracle(rt)
    assert same(_chain(dev, tris, dev.geom_build(tris), opt, W, H, cam, moves=True).accum, a.accum)
    assert same(_fused(rt, c, tris, opt, W, H, cam, moves=True), a.accum)
    b = _chain(spec, tris, gp, opt, W, H, cam, frames=4)
    assert same(_fused(rt, c, tris, opt, W, H, cam, frames=4, overlap=True), b.accum)
    spec.geom_free(gp)


def test_switching_off_renders_what_a_fresh_context_renders(rt, c):
    tris = lit_blocks_ao()
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    rt.set_light_tiles(7, 10)
    t = _fused(rt, c, tris, opt, 160, 90, CAM_AO)
    rt.set_light_tiles(0, 0)
    u = _fused(rt, c, tris, opt, 160, 90, CAM_AO)
    fresh = c.Runtime(0, c.MATH_EXACT)
    f = _fused(fresh, c, tris, opt, 160, 90, CAM_AO)
    fresh.close()
    assert same(u, f) and not same(t, u)


def test_refusals(rt, c):
    for bad in ((-1, 4), (4, -1), (17, 0), (0, 17), (12, 11)):
        with pytest.raises(c.CrtError, match="error %d: crt_set_light_tiles: .*log2_tile" % EINVAL):
            rt.set_light_tiles(*bad)
    tris = lit_blocks_ao()
    d_t, d_l = rt.to_device(tris), rt.to_device(orc.light_indices(tris))
    g = rt.build_geometry(d_t)
    with pytest.raises(c.CrtError, match="error %d: .*light tiles are off" % EINVAL):
        rt.light_tiles(g, d_l, 1)
    g.destroy()


@pytest.mark.parametrize("math", ["EXACT", "REFERENCE", "FAST"])
def test_row_ranges_equal_one_context(c, math):
    """three contexts, each rendering a band of rows (temporal reuse, no spatial reuse), give one context's rows"""
    tris = scene("blocks_restir")
    W, H = 192, 108
    opt = c.Options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=0)

    def render(y0, y1):
        r = c.Runtime(0, getattr(c, "MATH_" + math))
        r.set_light_sampling(c.LIGHTS_POWER)
        r.set_light_tiles(5, 8)
        r.set_row_range(y0, y1)
        app = c.RestirDI(r, W, H, tris, *CAM_RESTIR, opt, fused=True)
        for _ in range(3):
            app.frame()
        acc = app.accumulation.to_host().view(np.float32).reshape(H, W, 4)[::-1]
        app.geom.destroy()
        r.close()
        return acc

    whole = render(0, H)
    for y0, y1 in ((0, 37), (37, 71), (71, H)):
        assert same(render(y0, y1)[y0:y1], whole[y0:y1]), (y0, y1)


def test_slab_group_equals_one_slab():
    import torch

    import cedecrt as c
    import slabs

    tris = scene("blocks_restir")
    W, H = 960, 540
    torch.cuda.set_device(0)
    with torch.cuda.stream(torch.cuda.Stream()):
        part = slabs.SlabGroup(torch, None, 0, 1, tris, CAM_RESTIR, W, H, sub=3, overlap=True)
        full = slabs.SlabRenderer(torch, None, 0, 1, tris, CAM_RESTIR, W, H, fused=True)
        for r in (part, full):
            r.set_light_sampling(c.LIGHTS_POWER)
            r.set_light_tiles(7, 10)
        for _ in range(4):
            part.frame()
            full.frame()
        part.join()
        torch.cuda.synchronize()
        part.check()
        for sl in part.slabs:
            for name, elem in (("t_acc", 16), ("t_pix", 4)):
                assert torch.equal(sl._rows(getattr(sl, name), elem, sl.y0, sl.y1),
                                   full._rows(getattr(full, name), elem, sl.y0, sl.y1)), (name, sl.rank)
        part.close()


def _frame_means(rt, c, tris, mode, tiles, F, W=96, H=64, cam=CAM_FLOOR):
    """F independent frames of RIS without reuse: the mean of each frame's image over the lit pixels"""
    rt.set_light_sampling(mode, 0)
    rt.set_light_tiles(*tiles)
    opt = c.Options(accumulate=0, use_temporal_resampling=0, use_spatial_resampling=0)
    app = c.RestirDI(rt, W, H, tris, *cam, opt, fused=True)
    img = np.zeros((F, W * H, 3), np.float32)
    for f in range(F):
        app.frame()
        img[f] = app.accumulation.to_host().view(np.float32).reshape(-1, 4)[:, :3]
    app.geom.destroy()
    return img


@pytest.mark.parametrize("source", ["power", "uniform"])
def test_tiles_are_unbiased(rt, c, source):
    """selection with two tiles of 64 records (every tile shared by many pixels) against the same selection without
    tiles: the per-frame means over the lit region agree within z < 4"""
    tris = one_bright_many_dim()
    rt.set_math_mode(c.MATH_REFERENCE)
    mode = c.LIGHTS_POWER if source == "power" else c.LIGHTS_UNIFORM
    F = 256
    a, b = _frame_means(rt, c, tris, mode, (0, 0), F), _frame_means(rt, c, tris, mode, (1, 6), F)
    lit = np.concatenate([a, b]).mean(0).sum(1) > 0
    ma, mb = a[:, lit].mean(axis=(1, 2)), b[:, lit].mean(axis=(1, 2))
    z = abs(ma.mean() - mb.mean()) / np.sqrt(ma.var(ddof=1) / F + mb.var(ddof=1) / F)
    print("%s, tiles (1, 6) against none: z = %.2f, means %.5g / %.5g" % (source, z, ma.mean(), mb.mean()))
    assert z < 4  # measured on a B200: 0.47 (power), 2.22 (uniform); dividing by 1/S instead of the record's pdf: 284
