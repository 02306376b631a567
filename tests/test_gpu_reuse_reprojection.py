"""Unbiased reuse weights with a moving camera on the GPU (crt_temporal_resampling_reprojected_surfaces,
crt_restir_set_previous_frame): the launch list (typed call and crt_launch name) and the fused frame bit for bit against
the CPU specification in EXACT mode with a camera that moves twice (uniform and power light selection, the shadowed target
function on the per-kernel path), row ranges, the refusals of the new calls, and unbiasedness against plain RIS with the
camera stepping towards its final view."""
import ctypes as C

import numpy as np
import pytest

import orc
from helpers import DeviceAsOracle, same, small_scene
from test_gpu_reuse_weights import CAM_RIDGES, _last_frames, ridged_floor
from test_reuse_reprojection import MOVES, SurfacesChain, build_spec, moving
from test_reuse_weights import SCENES, VARIANTS, lit_blocks_ao

pytestmark = pytest.mark.gpu


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
    rt.set_reuse_weights(cedecrt.REUSE_REFERENCE)
    rt.set_light_sampling(cedecrt.LIGHTS_UNIFORM)
    rt.restir_set_previous_frame(None, None)


@pytest.fixture(scope="module")
def spec_lib():
    return build_spec()


@pytest.fixture()
def spec(spec_lib):
    """the CPU specification (tests/reuse/reuse_port_reprojected.cpp) in exact math"""
    s = spec_lib
    s.set_math_mode(1)
    yield s
    s.set_reuse_weights(0)
    s.set_light_sampling(0, 0)
    s.set_math_mode(0)


class DeviceSurfaces(DeviceAsOracle):
    """DeviceAsOracle with crt_temporal_resampling_reprojected_surfaces, called as a typed export or by_name through
    crt_launch"""

    def __init__(self, rt, by_name=False):
        super().__init__(rt)
        self.by_name = by_name

    def temporal_resampling_reprojected_surfaces(self, W, H, frame, g, tris, vis, eye, opt, prev_rg, prev_vis, prev, res):
        d_v, d_pv, d_p, d_r = (self.rt.to_device(a) for a in (vis, prev_vis, prev, res))
        if self.by_name:
            self.rt.launch("temporal_resampling_reprojected_surfaces", W, H, frame, g, g.triangles, d_v,
                           self.c.Float3(*[float(v) for v in eye]), self._opt(opt), self._rg(prev_rg), d_pv, d_p, d_r)
        else:
            self.rt.temporal_resampling_reprojected_surfaces(W, H, frame, g, g.triangles, d_v, tuple(eye), self._opt(opt),
                                                             self._rg(prev_rg), d_pv, d_p, d_r)
        res[:] = d_r.to_host()
        return res


def _app(rt, c, tris, opt, W, H, cam, name, fused):
    """cedecrt.RestirDI(reproject="surfaces") through the same camera path as moving(); the accumulation"""
    app = c.RestirDI(rt, W, H, tris, *cam, c.Options.from_numpy(opt), fused=fused, reproject="surfaces")
    for _ in range(2):
        app.frame()
    for eye, center in MOVES[name]:
        app.set_camera(eye, center)
        app.frame()
    acc = app.accumulation.to_host().view(np.float32).reshape(-1, 4)
    app.geom.destroy()
    return acc


@pytest.mark.parametrize("lights", ["uniform", "power"])
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_exact_moving_camera_equals_the_specification(rt, c, spec, name, lights):
    """the launch list (typed call and crt_launch name) and RestirDI(reproject="surfaces") — launch list, and fused frame
    with crt_restir_set_previous_frame, which takes the per-kernel path for the shadowed target function — against the
    specification bit for bit, 4 frames with a camera that moves twice"""
    make, W, H, cam = SCENES[name]
    W, H = 4 * W, 4 * H
    tris = make()
    power = lights == "power"
    spec.set_light_sampling(1 if power else 0, 0)
    spec.set_reuse_weights(1)
    rt.set_light_sampling(c.LIGHTS_POWER if power else c.LIGHTS_UNIFORM)
    rt.set_reuse_weights(c.REUSE_UNBIASED)
    gp = spec.geom_build(tris)
    for kw in VARIANTS:
        opt = orc.make_options(**kw)
        a = moving(SurfacesChain(spec, W, H, tris, gp, *cam, opt), name)
        assert float(a.accum[:, :3].sum()) > 0
        for by_name in (False, True):
            dev = DeviceSurfaces(rt, by_name)
            b = moving(SurfacesChain(dev, W, H, tris, dev.geom_build(tris), *cam, opt), name)
            assert same(a.accum, b.accum) and same(a.out, b.out) and same(a.temporal, b.temporal), (kw, by_name)
            for g in dev._geoms:
                g.destroy()
        for fused in (False, True):
            assert same(_app(rt, c, tris, opt, W, H, cam, name, fused), a.accum), (kw, fused)
    spec.geom_free(gp)


def test_row_ranges_with_a_moving_camera(c):
    """three contexts render bands of one image through the new launch-list call (every context reads the whole previous
    Visibility and history, written by all of them) with spatial reuse on and a camera that moves twice: equal to one
    context"""
    tris = small_scene("cornellbox1")
    W, H, cam = 192, 108, SCENES["cornellbox1"][3]
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)

    def render(bands):
        rts = []
        for y0, y1 in bands:
            r = c.Runtime(0, c.MATH_EXACT)
            r.set_reuse_weights(c.REUSE_UNBIASED)
            r.set_row_range(y0, y1)
            rts.append(r)
        per = []
        for r in rts:
            d_t = r.to_device(tris)
            per.append((r, d_t, r.build_geometry(d_t), r.to_device(orc.light_indices(tris))))
        r0 = rts[0]
        n = W * H
        vis, pvis = r0.buffer(c.VISIBILITY, n), r0.buffer(c.VISIBILITY, n)
        b0, b1 = r0.buffer(c.RESERVOIR, n), r0.buffer(c.RESERVOIR, n)
        temporal, acc = r0.buffer(c.RESERVOIR, n).zero(), r0.buffer(c.FLOAT4, n)
        o = c.Options.from_numpy(opt)

        def stage(fn):
            for r, d_t, g, d_l in per:
                fn(r, d_t, g, d_l)
            for r in rts:
                r.sync()

        cams = [cam, cam] + MOVES["cornellbox1"]
        prev_rg = None
        for f, (e, ctr) in enumerate(cams, 1):
            rg, eye = c.lookat(e, ctr, W, H), tuple(float(np.float32(v)) for v in e)
            vis, pvis = pvis, vis
            for r in rts:
                r.clear(acc, W, H)
            stage(lambda r, t, g, l: r.raycast(W, H, g, t, rg, vis))
            stage(lambda r, t, g, l: r.generate_candidate(W, H, f, g, t, vis, eye, l, o, b0))
            if prev_rg is None:
                stage(lambda r, t, g, l: r.temporal_resampling(W, H, f, g, t, vis, eye, o, temporal, b0))
            else:
                stage(lambda r, t, g, l: r.temporal_resampling_reprojected_surfaces(W, H, f, g, t, vis, eye, o, prev_rg,
                                                                                    pvis, temporal, b0))
            prev_rg = rg
            stage(lambda r, t, g, l: r.save_temporal_reservoir(W, H, b0, temporal))
            bi, bo = b0, b1
            for k in range(int(opt["spatial_resampling_passes"])):
                if k:
                    bi, bo = bo, bi
                stage(lambda r, t, g, l: r.spatial_resampling(W, H, f, k, g, t, vis, eye, o, bi, bo))
            stage(lambda r, t, g, l: r.resolve(acc, W, H, g, t, vis, eye, o, bo))
        out = acc.to_host().view(np.float32).reshape(-1, 4).copy(), bo.to_host().copy(), temporal.to_host().copy()
        for r, _, g, _ in per:
            g.destroy()
        for r in rts:
            r.close()
        return out

    whole = render([(0, H)])
    bands = render([(0, 37), (37, 71), (71, H)])
    assert all(same(x, y) for x, y in zip(whole, bands))
    assert float(whole[0][:, :3].sum()) > 0


def test_refusals_of_the_new_calls(rt, c):
    tris = lit_blocks_ao()
    cam = ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0))
    W, H, n = 64, 36, 64 * 36
    rt.set_reuse_weights(c.REUSE_UNBIASED)
    d_t = rt.to_device(tris)
    g = rt.build_geometry(d_t)
    rg, eye, o = c.lookat(*cam, W, H), tuple(float(np.float32(v)) for v in cam[0]), c.Options(use_temporal_resampling=1)
    vis, pvis, small = rt.buffer(c.VISIBILITY, n), rt.buffer(c.VISIBILITY, n), rt.buffer(c.VISIBILITY, n - 1)
    prev, res = rt.buffer(c.RESERVOIR, n).zero(), rt.buffer(c.RESERVOIR, n).zero()
    rt.raycast(W, H, g, d_t, rg, vis)
    rt.raycast(W, H, g, d_t, rg, pvis)
    with pytest.raises(c.CrtError, match="previous visibility buffer too small"):
        rt.temporal_resampling_reprojected_surfaces(W, H, 1, g, d_t, vis, eye, o, rg, small, prev, res)
    with pytest.raises(c.CrtError, match="Visibility must be a buffer of its own"):
        rt.temporal_resampling_reprojected_surfaces(W, H, 1, g, d_t, vis, eye, o, rg, vis, prev, res)
    with pytest.raises(c.CrtError, match="cannot run in place"):
        rt.temporal_resampling_reprojected_surfaces(W, H, 1, g, d_t, vis, eye, o, rg, pvis, res, res)
    with pytest.raises(c.CrtError, match="previous visibility buffer too small"):
        rt.launch("temporal_resampling_reprojected_surfaces", W, H, 1, g, d_t, vis, c.Float3(*eye), o, rg, small, prev, res)
    rt.temporal_resampling_reprojected_surfaces(W, H, 1, g, d_t, vis, eye, o, rg, pvis, prev, res)  # accepted
    g.destroy()
    # the fused frame: the stored Visibility must hold W * H records and must not be the frame's own
    app = c.RestirDI(rt, W, H, tris, *cam, c.Options(use_temporal_resampling=1), fused=True)
    app.frame()
    rt.restir_set_previous_frame(rg, small)
    with pytest.raises(c.CrtError, match="previous visibility buffer too small"):
        app.frame()
    rt.restir_set_previous_frame(rg, app.visibility)
    with pytest.raises(c.CrtError, match="Visibility must be a buffer of its own"):
        app.frame()
    rt.restir_set_previous_frame(rg, pvis)
    app.frame()  # accepted
    # crt_restir_set_previous_camera clears the stored Visibility: a camera without surfaces is refused again
    rt.set_reuse_weights(c.REUSE_REFERENCE)
    rt.restir_set_previous_camera(rg)
    rt.set_reuse_weights(c.REUSE_UNBIASED)
    with pytest.raises(c.CrtError, match="previous camera"):
        app.frame()
    # the fused frame on a row range narrower than the image stays refused
    rt.restir_set_previous_frame(rg, pvis)
    rt.set_row_range(0, H // 2)
    with pytest.raises(c.CrtError, match="whole image"):
        app.frame()
    rt.set_row_range(0, -1)
    rt.restir_set_previous_frame(None, None)
    app.geom.destroy()


# ---------------------------------------------------------------- unbiasedness
STEP = np.array([1.2, 0.6, -0.8])  # per frame; the chains' four eyes end at CAM_RIDGES


def _moving_chains(rt, c, tris, mode, N, W=128, H=96):
    """N independent chains of 4 frames (history zeroed, disjoint frame numbers, temporal + 3 spatial passes, no
    accumulation) whose camera steps towards CAM_RIDGES and ends there, with reprojection onto the previous frame's
    surfaces; the lit faces' region mean of each chain's last frame"""
    rt.set_reuse_weights(mode)
    opt = c.Options(accumulate=0, use_temporal_resampling=1, use_spatial_resampling=1)
    eye0, center = np.array(CAM_RIDGES[0]), CAM_RIDGES[1]
    app = c.RestirDI(rt, W, H, tris, *CAM_RIDGES, opt, fused=True, reproject="surfaces")
    means = []
    for _ in range(N):
        app.temporal.zero()
        app.prev_raygen = None
        for k in (3, 2, 1, 0):
            app.set_camera(tuple(eye0 + k * STEP), center)
            app.frame()
        means.append(app.accumulation.to_host().view(np.float32).reshape(-1, 4)[:, :3].astype(np.float64))
    app.geom.destroy()
    return means


def test_unbiased_reprojected_reuse_matches_plain_ris(rt, c):
    """the point of the feature.  The ridged floor of test_gpu_reuse_weights, 96 chains whose camera moves every frame
    against 96 frames of plain RIS at the final view; region means over the lit faces, z-score of the difference from the
    across-chain variance.  Bars: unbiased + reprojection z < 4; reference + reprojection z > 10 (the test sees bias).
    Measured on a B200 (1000 W power limit), N = 96: unbiased z = 0.23 (+0.03 %); reference z = 547, 51.5 % darker."""
    rt.set_math_mode(c.MATH_REFERENCE)
    tris = ridged_floor()
    N = 96
    ris, lit = _last_frames(rt, c, tris, False, c.REUSE_REFERENCE, N)
    assert 0.3 < lit.mean() < 0.7 and ris.mean() > 0
    z, rel = {}, {}
    for mode in (c.REUSE_UNBIASED, c.REUSE_REFERENCE):
        m = np.array([a[lit].sum(1).mean() for a in _moving_chains(rt, c, tris, mode, N)])
        z[mode] = abs(m.mean() - ris.mean()) / np.sqrt(m.var(ddof=1) / N + ris.var(ddof=1) / N)
        rel[mode] = m.mean() / ris.mean() - 1.0
    print("ridged floor, moving camera: unbiased z = %.2f (%+.4f), reference z = %.2f (%+.4f)"
          % (z[c.REUSE_UNBIASED], rel[c.REUSE_UNBIASED], z[c.REUSE_REFERENCE], rel[c.REUSE_REFERENCE]))
    assert z[c.REUSE_UNBIASED] < 4
    assert z[c.REUSE_REFERENCE] > 10
