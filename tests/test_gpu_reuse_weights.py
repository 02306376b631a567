"""Unbiased reuse weights on the GPU (crt_set_reuse_weights, CRT_REUSE_UNBIASED): the launch list and the fused frame bit
for bit against the CPU specification in EXACT mode (uniform and power light selection), the default unchanged after a
switch, row ranges through the per-kernel path, the refused combinations, and unbiasedness against plain RIS on a scene
built to show the reference's darkening."""
import numpy as np
import pytest

import orc
from helpers import DeviceAsOracle, same, small_scene
from test_light_sampling import light_port  # noqa: F401  (the fixture test_reuse_weights' reuse_port builds on)
from test_reuse_weights import SCENES, VARIANTS, _chain, lit_blocks_ao, reuse_port  # noqa: F401

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


@pytest.fixture()
def spec(reuse_port):  # noqa: F811
    """the CPU specification (tests/reuse/reuse_port.cpp) in exact math"""
    reuse_port.set_math_mode(1)
    yield reuse_port
    reuse_port.set_reuse_weights(0)
    reuse_port.set_light_sampling(0, 0)
    reuse_port.set_math_mode(0)


def _fused(rt, c, tris, opt, W, H, cam, frames=3):
    app = c.RestirDI(rt, W, H, tris, *cam, c.Options.from_numpy(opt), fused=True)
    for _ in range(frames):
        app.frame()
    acc = app.accumulation.to_host().view(np.float32).reshape(-1, 4)
    app.geom.destroy()
    return acc


@pytest.mark.parametrize("lights", ["uniform", "power"])
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_exact_unbiased_equals_the_specification(rt, c, spec, name, lights):
    """the launch list (per-kernel path) and the fused frame, 3 frames, against the specification bit for bit; the
    shadowed target function on the per-kernel path only (the fused frame falls back to it)"""
    make, W, H, cam = SCENES[name]
    W, H = 4 * W, 4 * H
    tris = make()
    power = lights == "power"
    spec.set_light_sampling(1 if power else 0, 0)
    spec.set_reuse_weights(1)
    rt.set_light_sampling(c.LIGHTS_POWER if power else c.LIGHTS_UNIFORM)
    rt.set_reuse_weights(c.REUSE_UNBIASED)
    dev = DeviceAsOracle(rt)
    gp, gd = spec.geom_build(tris), dev.geom_build(tris)
    for kw in VARIANTS:
        opt = orc.make_options(**kw)
        a, b = _chain(spec, tris, gp, opt, W, H, cam), _chain(dev, tris, gd, opt, W, H, cam)
        assert same(a.accum, b.accum) and same(a.out, b.out) and same(a.temporal, b.temporal), kw
        if not kw.get("use_shadowed_target_function"):
            assert same(_fused(rt, c, tris, opt, W, H, cam), a.accum), kw
    spec.geom_free(gp)


def test_switching_back_renders_what_a_fresh_context_renders(rt, c):
    tris = lit_blocks_ao()
    cam = ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0))
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    dev = DeviceAsOracle(rt)
    gd = dev.geom_build(tris)
    rt.set_reuse_weights(c.REUSE_UNBIASED)
    u = (_fused(rt, c, tris, opt, 160, 90, cam), _chain(dev, tris, gd, opt, 160, 90, cam).accum)
    rt.set_reuse_weights(c.REUSE_REFERENCE)
    r = (_fused(rt, c, tris, opt, 160, 90, cam), _chain(dev, tris, gd, opt, 160, 90, cam).accum)
    fresh = c.Runtime(0, c.MATH_EXACT)
    fdev = DeviceAsOracle(fresh)
    f = (_fused(fresh, c, tris, opt, 160, 90, cam), _chain(fdev, tris, fdev.geom_build(tris), opt, 160, 90, cam).accum)
    fresh.close()
    assert same(r[0], f[0]) and same(r[1], f[1])
    assert not same(u[0], r[0]) and not same(u[1], r[1])


def _banded_launch_list(c, tris, W, H, cam, opt, bands, frames=3):
    """one context per band of rows, every context writing into the same device buffers (those of the first), one stage
    at a time: every context finishes a stage, synchronised, before any context starts the next"""
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
    vis, b0, b1 = r0.buffer(c.VISIBILITY, n), r0.buffer(c.RESERVOIR, n), r0.buffer(c.RESERVOIR, n)
    temporal, acc = r0.buffer(c.RESERVOIR, n).zero(), r0.buffer(c.FLOAT4, n)
    for r in rts:
        r.clear(acc, W, H)
    rg, eye, o = c.lookat(*cam, W, H), tuple(float(np.float32(v)) for v in cam[0]), c.Options.from_numpy(opt)

    def stage(fn):
        for r, d_t, g, d_l in per:
            fn(r, d_t, g, d_l)
        for r in rts:
            r.sync()

    for f in range(1, frames + 1):
        stage(lambda r, t, g, l: r.raycast(W, H, g, t, rg, vis))
        stage(lambda r, t, g, l: r.generate_candidate(W, H, f, g, t, vis, eye, l, o, b0))
        stage(lambda r, t, g, l: r.temporal_resampling(W, H, f, g, t, vis, eye, o, temporal, b0))
        stage(lambda r, t, g, l: r.save_temporal_reservoir(W, H, b0, temporal))
        bi, bo = b0, b1
        for k in range(int(opt["spatial_resampling_passes"])):
            if k:
                bi, bo = bo, bi
            stage(lambda r, t, g, l: r.spatial_resampling(W, H, f, k, g, t, vis, eye, o, bi, bo))
        stage(lambda r, t, g, l: r.resolve(acc, W, H, g, t, vis, eye, o, bo))
    out = acc.to_host().view(np.float32).reshape(-1, 4).copy(), bo.to_host().copy()
    for r, _, g, _ in per:
        g.destroy()
    for r in rts[1:]:
        r.close()
    return out, r0


def test_row_ranges_through_the_per_kernel_path(c):
    """three contexts render bands of one image through the launch list with spatial reuse on: equal to one context"""
    tris = small_scene("cornellbox1")
    W, H, cam = 192, 108, ((0.0, 2.7, 9.0), (0.0, 2.7, 0.0))
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    (whole_acc, whole_res), r = _banded_launch_list(c, tris, W, H, cam, opt, [(0, H)])
    r.close()
    (band_acc, band_res), r = _banded_launch_list(c, tris, W, H, cam, opt, [(0, 37), (37, 71), (71, H)])
    r.close()
    assert same(band_acc, whole_acc) and same(band_res, whole_res)
    assert float(whole_acc[:, :3].sum()) > 0


def test_refused_combinations(rt, c):
    tris = lit_blocks_ao()
    cam = ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0))
    W, H = 64, 36
    with pytest.raises(c.CrtError, match="unknown reuse weight mode"):
        rt.set_reuse_weights(2)
    rt.set_reuse_weights(c.REUSE_UNBIASED)
    # a previous camera: the launch list's reprojected temporal merge and the fused frame's
    with pytest.raises(c.CrtError, match="previous camera"):
        app = c.RestirDI(rt, W, H, tris, *cam, c.Options(use_temporal_resampling=1), fused=False, reproject=True)
        for _ in range(2):
            app.frame()
    app.geom.destroy()
    with pytest.raises(c.CrtError, match="previous camera"):
        app = c.RestirDI(rt, W, H, tris, *cam, c.Options(use_temporal_resampling=1), fused=True, reproject=True)
        for _ in range(2):
            app.frame()
    app.geom.destroy()
    # a previous camera set before the switch: refused by the frame
    rt.set_reuse_weights(c.REUSE_REFERENCE)
    rt.restir_set_previous_camera(c.lookat(*cam, W, H))
    rt.set_reuse_weights(c.REUSE_UNBIASED)
    app = c.RestirDI(rt, W, H, tris, *cam, c.Options(use_temporal_resampling=1), fused=True)
    with pytest.raises(c.CrtError, match="previous camera"):
        app.frame()
    rt.restir_set_previous_camera(None)
    app.frame()  # no camera: accepted
    # the fused frame on a row range narrower than the image; the per-kernel path takes it
    rt.set_row_range(0, H // 2)
    with pytest.raises(c.CrtError, match="whole image"):
        app.frame()
    shadowed = c.RestirDI(rt, W, H, tris, *cam, c.Options(use_shadowed_target_function=1, use_spatial_resampling=0),
                          fused=True)
    shadowed.frame()
    rt.set_row_range(0, -1)
    app.geom.destroy()
    shadowed.geom.destroy()


# ---------------------------------------------------------------- unbiasedness
def ridged_floor(seed=5, n_ridges=24, width=24.0):
    """a sawtooth floor along x (faces tilted about +-15 degrees, seeded jitter) under a low area light far along +x, so
    that about half the faces (those tilted away) have the light below their horizon"""
    rng = np.random.default_rng(seed)
    xs = np.linspace(-width / 2, width / 2, 2 * n_ridges + 1)
    xs[1:-1] += rng.uniform(-0.1, 0.1, len(xs) - 2) * (xs[1] - xs[0])
    h = np.tan(np.radians(15.0)) * (xs[1] - xs[0])
    ys = np.where(np.arange(len(xs)) % 2 == 0, 0.0, h)
    z0, z1 = -width / 2, width / 2
    tris = []
    for i in range(len(xs) - 1):
        a, b = (xs[i], ys[i]), (xs[i + 1], ys[i + 1])
        q = [[a[0], a[1], z0], [b[0], b[1], z0], [b[0], b[1], z1], [a[0], a[1], z1]]
        tris += [(q[0], q[2], q[1]), (q[0], q[3], q[2])]
    out = np.zeros(len(tris) + 2, orc.TRIANGLE)
    out["vertices"][:len(tris)] = np.array(tris, np.float32)
    out["color"][:len(tris)] = 0.6
    L = [[40.0, 1.5, -8.0], [40.0, 1.5, 8.0], [40.0, 6.0, 8.0], [40.0, 6.0, -8.0]]  # 2-12 degrees above the floor
    out["vertices"][-2] = [L[0], L[1], L[2]]
    out["vertices"][-1] = [L[0], L[2], L[3]]
    out["emissive"][-2:] = (400.0, 380.0, 360.0)
    return out


CAM_RIDGES = ((0.0, 14.0, 10.0), (0.0, 0.0, 0.0))


def _last_frames(rt, c, tris, reuse, mode, N, W=128, H=96):
    """N independent values of the lit faces' region mean: with reuse, N chains of 4 frames (history zeroed, disjoint
    frame numbers, temporal + 3 spatial passes, no accumulation) keeping the last frame; without, N frames of plain RIS"""
    rt.set_reuse_weights(mode)
    opt = c.Options(accumulate=0, use_temporal_resampling=int(reuse), use_spatial_resampling=int(reuse))
    app = c.RestirDI(rt, W, H, tris, *CAM_RIDGES, opt, fused=True)
    app.frame()
    vis = app.visibility.to_host()
    idx = vis["index"]
    v = tris["vertices"][np.maximum(idx, 0)].astype(np.float64)
    nx = np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0])[:, 0]
    lit = (idx >= 0) & (idx < len(tris) - 2) & (nx > 0)  # faces tilted towards +x: the light above their horizon
    means = []
    for _ in range(N):
        if reuse:
            app.temporal.zero()
            for _ in range(3):
                app.frame()
        app.frame()
        a = app.accumulation.to_host().view(np.float32).reshape(-1, 4)[:, :3].astype(np.float64)
        means.append(a[lit].sum(1).mean())
    app.geom.destroy()
    return np.array(means), lit


def test_unbiased_reuse_matches_plain_ris_where_the_reference_darkens(rt, c):
    """the point of the feature.  On the ridged floor the reference's reuse darkens the lit faces: a lit pixel merges
    neighbours on faces whose samples are occluded (visibility reuse zeroes their weight but keeps their M) and whose M
    counts although the 1/M normalisation has nothing to correct for.  Region means over the lit faces, z-score of the
    difference to plain RIS from the across-chain variance.  Measured on a B200 (1000 W power limit), N = 96:
    unbiased z = 0.14 (+0.01 %); reference z = 526, 48.8 % darker."""
    rt.set_math_mode(c.MATH_REFERENCE)
    tris = ridged_floor()
    N = 96
    ris, lit = _last_frames(rt, c, tris, False, c.REUSE_REFERENCE, N)
    assert 0.3 < lit.mean() < 0.7 and ris.mean() > 0
    z, rel = {}, {}
    for mode in (c.REUSE_UNBIASED, c.REUSE_REFERENCE):
        m, _ = _last_frames(rt, c, tris, True, mode, N)
        z[mode] = abs(m.mean() - ris.mean()) / np.sqrt(m.var(ddof=1) / N + ris.var(ddof=1) / N)
        rel[mode] = m.mean() / ris.mean() - 1.0
    print("ridged floor: unbiased z = %.2f (%+.4f), reference z = %.2f (%+.4f)"
          % (z[c.REUSE_UNBIASED], rel[c.REUSE_UNBIASED], z[c.REUSE_REFERENCE], rel[c.REUSE_REFERENCE]))
    assert z[c.REUSE_UNBIASED] < 4
    assert z[c.REUSE_REFERENCE] > 10 and rel[c.REUSE_REFERENCE] < 0
