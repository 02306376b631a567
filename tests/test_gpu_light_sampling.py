"""Power-proportional light selection on the GPU (crt_set_light_sampling, CRT_LIGHTS_POWER): the device's slot table
against the port's byte for byte, every light-sampling path bit for bit against the port in EXACT mode, the identity
n = K = 2^k (power == uniform), unbiasedness and noise against uniform selection, invalidation, and the error cases."""
import os

import numpy as np
import pytest

import orc
from helpers import DeviceAsOracle, same, scene, small_scene
from test_light_sampling import light_port, light_set  # noqa: F401  (light_port: the fixture)

pytestmark = pytest.mark.gpu
CAM_AO = ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0))


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
    rt.set_light_sampling(cedecrt.LIGHTS_UNIFORM)
    yield cedecrt
    rt.set_light_sampling(cedecrt.LIGHTS_UNIFORM)


@pytest.fixture()
def port1(light_port):
    """the CPU specification (tests/lights/light_port.cpp) in exact math"""
    light_port.set_math_mode(1)
    yield light_port
    light_port.set_light_sampling(0, 0)
    light_port.set_math_mode(0)


def lit_blocks_ao(n_lights=64, seed=3):
    tris = small_scene("blocks_ao").copy()
    tris["emissive"][100:100 + n_lights] = np.random.default_rng(seed).uniform(0.5, 30.0, (n_lights, 3))
    return tris


def device_table(rt, tris, lights, mode, log2):
    d_t, d_l = rt.to_device(tris), rt.to_device(lights)
    g = rt.build_geometry(d_t)
    rt.set_light_sampling(mode, log2)
    try:
        return rt.light_sampling_table(g, d_l)
    finally:
        g.destroy()


TABLE_CASES = [("lit_blocks_ao", 0), ("lit_blocks_ao", 12), ("odd", 0), ("odd", 11), ("one", 0), ("equal", 0),
               ("dominant", 17), ("blocks_restir", 0), ("big", 0)]


@pytest.mark.parametrize("name,log2", TABLE_CASES)
def test_table_equals_port(rt, c, port1, name, log2):
    if name == "lit_blocks_ao":
        tris = lit_blocks_ao()
        lights = orc.light_indices(tris)
    elif name == "blocks_restir":  # the stand-in, ~146 k lights: K = 2^20
        tris = scene("blocks_restir")
        lights = orc.light_indices(tris)
    elif name == "big":  # more than 2^22 lights: K = 2^23
        tris, lights = light_set(np.random.default_rng(5), (1 << 22) + 4099, "random")
    else:
        n = {"odd": 700, "one": 1, "equal": 64, "dominant": 1000}[name]
        tris, lights = light_set(np.random.default_rng(n + log2), n, name if name != "one" else "random")
    port1.set_light_sampling(1, log2)
    want, starts = port1.light_table(tris, lights)
    got = device_table(rt, tris, lights, c.LIGHTS_POWER, log2)
    assert same_up_to_nan_payload(got, want)


def same_up_to_nan_payload(a, b):
    """bit equality, except that a NaN equals a NaN: the normal of a zero-area light is 0/0, whose payload is the
    hardware's (x86 and the GPU produce different quiet NaNs)"""
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool((na == nb).all()) and same(np.where(na, 0, a), np.where(nb, 0, b))


def test_errors(rt, c):
    tris = lit_blocks_ao()
    lights = orc.light_indices(tris)
    with pytest.raises(c.CrtError):
        rt.set_light_sampling(2)
    with pytest.raises(c.CrtError):
        rt.set_light_sampling(c.LIGHTS_POWER, -1)
    for bad in (5, 24):  # 2^5 < 64 lights; above 2^23
        with pytest.raises(c.CrtError, match="log2_slots"):
            device_table(rt, tris, lights, c.LIGHTS_POWER, bad)
    many = np.resize(lights, (1 << 23) + 1)  # a light list may name a triangle more than once
    with pytest.raises(c.CrtError, match="2\\^23"):
        device_table(rt, tris, many, c.LIGHTS_POWER, 0)
    # uniform mode ignores the slot count
    assert len(device_table(rt, tris, lights, c.LIGHTS_UNIFORM, 5)) == 64


def _chain(o, tris, g, opt, W, H, moves=False, frames=3, cam=CAM_AO):
    ch = orc.RestirChain(o, W, H, tris, g, *cam, opt, reproject=moves)
    for f in range(frames):
        if moves and f:
            ch.set_camera((8.0 + 0.3 * f, 8.0, 8.0 - 0.2 * f), (0.0, 0.0, 0.0))
        ch.step()
    return ch


def _fused(rt, c, tris, opt, W, H, moves=False, frames=3, cam=CAM_AO):
    app = c.RestirDI(rt, W, H, tris, *cam, c.Options.from_numpy(opt), fused=True, reproject=moves)
    for f in range(frames):
        if moves and f:
            app.set_camera((8.0 + 0.3 * f, 8.0, 8.0 - 0.2 * f), (0.0, 0.0, 0.0))
        app.frame()
    acc = app.accumulation.to_host().view(np.float32).reshape(-1, 4)
    app.geom.destroy()
    return acc


def _paths(o, tris, g, example, opt, W, H, frames=2):
    rg = o.lookat(*CAM_AO, W, H)
    acc = np.zeros((W * H, 4), np.float32)
    for f in range(1, frames + 1):
        if o.kind == "cuda":
            o.path_trace(example, W, H, f, g, tris, orc.light_indices(tris), rg, opt, acc)
        else:
            o.set_example(example)
            o.path_trace(W, H, f, g, tris, orc.light_indices(tris), rg, opt, acc)
    return acc


SCENES = {"cornellbox1": (lambda: small_scene("cornellbox1"), 96, 54, ((0.0, 2.7, 9.0), (0.0, 2.7, 0.0))),
          "lit_blocks_ao": (lit_blocks_ao, 320, 180, CAM_AO)}


@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
@pytest.mark.parametrize("log2", [0, 10])
def test_restir_exact_power_mode_equals_port(rt, c, port1, name, log2):
    make, W, H, cam = SCENES[name]
    tris = make()
    port1.set_light_sampling(1, log2)
    rt.set_light_sampling(c.LIGHTS_POWER, log2)
    dev = DeviceAsOracle(rt)
    gp, gd = port1.geom_build(tris), dev.geom_build(tris)
    base = dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    for kw in (base, dict(base, use_shadowed_target_function=1), dict(base, use_visibility_reuse=0)):
        opt = orc.make_options(**kw)
        a, b = _chain(port1, tris, gp, opt, W, H, cam=cam), _chain(dev, tris, gd, opt, W, H, cam=cam)
        assert same(a.accum, b.accum) and same(a.out, b.out), kw  # the per-kernel launch list
        if not kw.get("use_shadowed_target_function"):
            assert same(_fused(rt, c, tris, opt, W, H, cam=cam), a.accum), kw  # the fused frame
    # a moving camera under reprojection
    opt = orc.make_options(**base)
    a = _chain(port1, tris, gp, opt, W, H, moves=True)
    assert same(_chain(dev, tris, gd, opt, W, H, moves=True).accum, a.accum)
    assert same(_fused(rt, c, tris, opt, W, H, moves=True), a.accum)
    port1.geom_free(gp)


def _wavefront_off_runtime(c):
    os.environ["CRT_WAVEFRONT"] = "0"
    try:
        return c.Runtime(0, c.MATH_EXACT)
    finally:
        del os.environ["CRT_WAVEFRONT"]


@pytest.mark.parametrize("example,shadowed", [(8, 0), (9, 0), (9, 1)])
def test_path_tracers_exact_power_mode_equals_port(rt, c, port1, example, shadowed):
    tris = lit_blocks_ao()
    W, H = 160, 90
    opt = orc.make_options(accumulate=1, max_depth=4, ris_sample_count=16, use_shadowed_target_function=shadowed)
    gp = port1.geom_build(tris)
    port1.set_light_sampling(1, 0)
    want = _paths(port1, tris, gp, example, opt, W, H)
    single = _wavefront_off_runtime(c)
    for r in (rt, single):
        r.set_light_sampling(c.LIGHTS_POWER, 0)
        dev = DeviceAsOracle(r)
        gd = dev.geom_build(tris)
        assert same(_paths(dev, tris, gd, example, opt, W, H), want), "wavefront" if r is rt else "CRT_WAVEFRONT=0"
    single.close()
    port1.geom_free(gp)


@pytest.mark.parametrize("math", ["EXACT", "REFERENCE"])
def test_power_equals_uniform_when_every_light_owns_one_slot(rt, c, math):
    """n = K = 2^k: c_i = 1 and sel_i = 1.0f / (float)n for every light, so every path computes the uniform mode's bits"""
    tris = lit_blocks_ao(64)
    W, H = 160, 90
    rt.set_math_mode(getattr(c, "MATH_" + math))
    dev = DeviceAsOracle(rt)
    gd = dev.geom_build(tris)
    restir = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    shadowed = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1, use_shadowed_target_function=1)
    single = _wavefront_off_runtime(c)
    single.set_math_mode(getattr(c, "MATH_" + math))
    sdev = DeviceAsOracle(single)
    sgd = sdev.geom_build(tris)
    out = {}
    for mode, log2 in ((c.LIGHTS_UNIFORM, 0), (c.LIGHTS_POWER, 6)):
        rt.set_light_sampling(mode, log2)
        single.set_light_sampling(mode, log2)
        r = [_fused(rt, c, tris, restir, W, H), _chain(dev, tris, gd, restir, W, H).accum, _chain(dev, tris, gd, shadowed, W, H).accum]
        for ex, sh in ((8, 0), (9, 0), (9, 1)):
            popt = orc.make_options(accumulate=1, max_depth=4, ris_sample_count=16, use_shadowed_target_function=sh)
            r += [_paths(dev, tris, gd, ex, popt, W, H), _paths(sdev, tris, sgd, ex, popt, W, H)]
        out[mode] = r
    single.close()
    for k, (u, p) in enumerate(zip(out[c.LIGHTS_UNIFORM], out[c.LIGHTS_POWER])):
        assert same(u, p), k


def test_switching_back_to_uniform_renders_what_a_fresh_context_renders(rt, c):
    tris = lit_blocks_ao()
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    rt.set_light_sampling(c.LIGHTS_POWER)
    p = _fused(rt, c, tris, opt, 160, 90)
    rt.set_light_sampling(c.LIGHTS_UNIFORM)
    u = _fused(rt, c, tris, opt, 160, 90)
    fresh = c.Runtime(0, c.MATH_EXACT)
    f = _fused(fresh, c, tris, opt, 160, 90)
    fresh.close()
    assert same(u, f) and not same(p, u)


def test_table_follows_refit_and_in_place_emission_changes(rt, c, port1):
    tris = lit_blocks_ao()
    lights = orc.light_indices(tris)
    d_t, d_l = rt.to_device(tris), rt.to_device(lights)
    g = rt.build_geometry(d_t)
    rt.set_light_sampling(c.LIGHTS_POWER, 0)
    port1.set_light_sampling(1, 0)
    assert same(rt.light_sampling_table(g, d_l), port1.light_table(tris, lights)[0])
    tris["vertices"][lights[5]] *= 1.5  # a bigger emitter: more power, more slots
    d_t.upload(tris)
    g.refit()
    assert same(rt.light_sampling_table(g, d_l), port1.light_table(tris, lights)[0])
    before = np.diff(port1.light_table(tris, lights)[1].astype(np.int64))[7]
    tris["emissive"][lights[7]] = (200.0, 200.0, 200.0)
    d_t.upload(tris)
    rt.lights_changed(g)
    got = rt.light_sampling_table(g, d_l)
    want = port1.light_table(tris, lights)
    assert same(got, want[0]) and np.diff(want[1].astype(np.int64))[7] > before
    g.destroy()


def one_bright_many_dim(seed=11, n_dim=1000):
    """a floor under one bright emitter and ~1000 dim ones (seeded)"""
    rng = np.random.default_rng(seed)
    n = 2 + 1 + n_dim
    tris = np.zeros(n, orc.TRIANGLE)
    tris["vertices"][0] = [[-20, 0, -20], [20, 0, -20], [20, 0, 20]]
    tris["vertices"][1] = [[-20, 0, -20], [20, 0, 20], [-20, 0, 20]]
    tris["color"][:2] = 0.7
    tris["vertices"][2] = [[-1, 6, -1], [1, 6, -1], [0, 6, 1.5]]
    tris["emissive"][2] = (60.0, 55.0, 50.0)
    p = rng.uniform([-15, 2, -15], [15, 9, 15], (n_dim, 3)).astype(np.float32)
    tris["vertices"][3:] = p[:, None, :] + rng.uniform(-0.15, 0.15, (n_dim, 3, 3)).astype(np.float32)
    tris["emissive"][3:] = rng.uniform(0.05, 0.3, (n_dim, 3))
    return tris


CAM_FLOOR = ((0.0, 14.0, 18.0), (0.0, 0.0, 0.0))


def _frames(rt, c, tris, which, mode, F, W=96, H=64, cam=CAM_FLOOR):
    """F independent frames (no accumulation, no reuse): per-frame linear images, shape (F, W*H, 3)"""
    rt.set_light_sampling(mode, 0)
    out = np.zeros((F, W * H, 3), np.float32)
    if which == "restir":
        opt = c.Options(accumulate=0, use_temporal_resampling=0, use_spatial_resampling=0)
        app = c.RestirDI(rt, W, H, tris, *cam, opt, fused=True)
        for f in range(F):
            app.frame()
            out[f] = app.accumulation.to_host().view(np.float32).reshape(-1, 4)[:, :3]
        app.geom.destroy()
        return out
    d_t, d_l = rt.to_device(tris), rt.to_device(orc.light_indices(tris))
    g = rt.build_geometry(d_t)
    acc = rt.buffer(c.FLOAT4, W * H)
    rg = c.lookat(*cam, W, H)
    opt = c.Options(accumulate=0, max_depth=2)
    for f in range(F):
        rt.path_trace(8, W, H, f + 1, g, d_t, d_l, rg, opt, acc)
        out[f] = acc.to_host().view(np.float32).reshape(-1, 4)[:, :3]
    g.destroy()
    return out


@pytest.mark.parametrize("which", ["nee", "restir"])
@pytest.mark.parametrize("scene_name", ["bright_and_dim", "blocks_restir"])
def test_power_mode_is_unbiased_and_less_noisy(rt, c, which, scene_name):
    if scene_name == "bright_and_dim":
        tris, cam, F = one_bright_many_dim(), CAM_FLOOR, 256
    else:  # a band of the stand-in's config-4/5 view
        tris, cam, F = scene("blocks_restir"), ((0.0, 22.0, 0.0), (30.0, 18.0, 30.0)), 64
    rt.set_math_mode(c.MATH_REFERENCE)
    img = {m: _frames(rt, c, tris, which, m, F, cam=cam) for m in (c.LIGHTS_UNIFORM, c.LIGHTS_POWER)}
    m = {k: v.mean(axis=(1, 2)) for k, v in img.items()}  # per-frame image means: independent samples
    u, p = m[c.LIGHTS_UNIFORM], m[c.LIGHTS_POWER]
    z = abs(u.mean() - p.mean()) / np.sqrt(u.var(ddof=1) / F + p.var(ddof=1) / F)
    ref = np.concatenate([img[c.LIGHTS_UNIFORM], img[c.LIGHTS_POWER]]).mean(0)
    mse = {k: float(((v[:16].mean(0) - ref) ** 2).mean() / (ref ** 2).mean()) for k, v in img.items()}
    ratio = mse[c.LIGHTS_POWER] / mse[c.LIGHTS_UNIFORM]
    print("%s %s: z = %.2f, relative MSE after 16 frames uniform %.3g power %.3g, ratio %.3f"
          % (scene_name, which, z, mse[c.LIGHTS_UNIFORM], mse[c.LIGHTS_POWER], ratio))
    assert z < 4  # measured on a B200: 1.28 / 0.25 (bright and dim, nee / restir), 0.01 / 0.38 (stand-in)
    if scene_name == "bright_and_dim":
        assert ratio < 1.0  # measured on a B200: 0.017 (nee), 0.016 (restir without reuse)


def test_row_slabs_equal_one_frame_in_power_mode(c):
    """three contexts, each rendering a band of rows with its own geometry and slot table, give the single context's
    rows (temporal reuse on; spatial reuse off, so no slab reads another's rows and no halo exchange is needed)"""
    tris = scene("blocks_restir")
    W, H, cam = 192, 108, ((0.0, 22.0, 0.0), (30.0, 18.0, 30.0))
    opt = c.Options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=0)

    def render(y0, y1):
        r = c.Runtime(0, c.MATH_EXACT)
        r.set_light_sampling(c.LIGHTS_POWER)
        r.set_row_range(y0, y1)
        app = c.RestirDI(r, W, H, tris, *cam, opt, fused=True)
        for _ in range(3):
            app.frame()
        acc = app.accumulation.to_host().view(np.float32).reshape(H, W, 4)[::-1]  # bottom-up buffer -> row yi
        app.geom.destroy()
        r.close()
        return acc

    whole = render(0, H)
    edges = [0, 37, 71, H]
    for y0, y1 in zip(edges[:-1], edges[1:]):
        assert same(render(y0, y1)[y0:y1], whole[y0:y1]), (y0, y1)
