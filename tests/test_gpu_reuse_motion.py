"""Reprojection that follows moving geometry on the GPU (crt_temporal_resampling_reprojected_motion,
crt_restir_set_previous_triangles, RestirDI.set_triangles): the launch list (typed call and crt_launch name) and RestirDI on
the launch list, the fused frame and its per-kernel path bit for bit against the CPU specification in EXACT mode while
triangles and camera move, with uniform and power light selection under both reuse weights; the identity in every math
mode; row ranges; frame overlap with the primary-ray prefetch; the refusals; and unbiasedness on a ridged floor whose
sawtooth flips every frame."""
import os

import numpy as np
import pytest

import orc
from helpers import DeviceAsOracle, same, scene, small_scene
from test_gpu_reuse_weights import CAM_RIDGES, _last_frames, ridged_floor
from test_reuse_motion import MotionChain, MotionPort, _build, animate, move_triangles
from test_reuse_reprojection import MOVES
from test_reuse_weights import REUSE, SCENES, VARIANTS, lit_blocks_ao

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
    rt.set_frame_overlap(0)


@pytest.fixture(scope="module")
def spec_lib():
    return _build("reuse_port_motion.cpp", os.path.join(REUSE, "libreuse_port_motion.so"), "c++20",
                  ["-ffp-contract=off", "-fno-fast-math"], MotionPort)


@pytest.fixture()
def spec(spec_lib):
    """the CPU specification (tests/reuse/reuse_port_motion.cpp) in exact math"""
    s = spec_lib
    s.set_math_mode(1)
    yield s
    s.set_reuse_weights(0)
    s.set_light_sampling(0, 0)
    s.set_math_mode(0)


class DeviceMotion(DeviceAsOracle):
    """DeviceAsOracle with the reprojected calls: crt_temporal_resampling_reprojected_motion as a typed export or by name
    through crt_launch, and crt_temporal_resampling_reprojected_surfaces"""

    def __init__(self, rt, by_name=False):
        super().__init__(rt)
        self.by_name = by_name

    def temporal_resampling_motion(self, W, H, frame, g, tris, vis, eye, opt, prev_rg, prev_tris, prev_vis, prev, res):
        d_v, d_pt, d_pv, d_p, d_r = (self.rt.to_device(a) for a in (vis, prev_tris, prev_vis, prev, res))
        if self.by_name:
            self.rt.launch("temporal_resampling_reprojected_motion", W, H, frame, g, g.triangles, d_v,
                           self.c.Float3(*[float(v) for v in eye]), self._opt(opt), self._rg(prev_rg), d_pt, d_pv, d_p, d_r)
        else:
            self.rt.temporal_resampling_reprojected_motion(W, H, frame, g, g.triangles, d_v, tuple(eye), self._opt(opt),
                                                           self._rg(prev_rg), d_pt, d_pv, d_p, d_r)
        res[:] = d_r.to_host()
        return res

    def temporal_resampling_reprojected_surfaces(self, W, H, frame, g, tris, vis, eye, opt, prev_rg, prev_vis, prev, res):
        d_v, d_pv, d_p, d_r = (self.rt.to_device(a) for a in (vis, prev_vis, prev, res))
        self.rt.temporal_resampling_reprojected_surfaces(W, H, frame, g, g.triangles, d_v, tuple(eye), self._opt(opt),
                                                         self._rg(prev_rg), d_pv, d_p, d_r)
        res[:] = d_r.to_host()
        return res


def _app(rt, c, scene, opt, W, H, cam, name, fused, reproject, moves=True, overlap=False):
    """RestirDI through animate()'s path: set_triangles (a refit) and set_camera before each moved frame; the accumulation"""
    app = c.RestirDI(rt, W, H, scene, *cam, c.Options.from_numpy(opt), fused=fused, reproject=reproject)
    if overlap:
        rt.set_frame_overlap(1)
        app.prefetch = True
    try:
        for _ in range(2):
            app.frame()
        for k, (eye, center) in enumerate(MOVES[name]):
            app.set_triangles(move_triangles(scene, k + 1) if moves else scene)
            app.set_camera(eye, center)
            app.frame()
        rt.frame_join()
        acc = app.accumulation.to_host().view(np.float32).reshape(-1, 4).copy()
    finally:
        rt.set_frame_overlap(0)
        app.geom.destroy()
    return acc


@pytest.mark.parametrize("reuse", [0, 1])
@pytest.mark.parametrize("lights", ["uniform", "power"])
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_exact_motion_equals_the_specification(rt, c, spec, name, lights, reuse):
    """the launch list (typed call and crt_launch name) and RestirDI with set_triangles — launch list, fused frame with
    crt_restir_set_previous_triangles, which takes the per-kernel path for the shadowed target function — against the
    specification bit for bit, 5 frames in which triangles and camera move twice; reproject=True under the reference's
    weights, "surfaces" under both"""
    make, W, H, cam = SCENES[name]
    W, H = 4 * W, 4 * H
    scene = make()
    power = lights == "power"
    spec.set_light_sampling(1 if power else 0, 0)
    spec.set_reuse_weights(reuse)
    rt.set_light_sampling(c.LIGHTS_POWER if power else c.LIGHTS_UNIFORM)
    rt.set_reuse_weights(c.REUSE_UNBIASED if reuse else c.REUSE_REFERENCE)
    for kw in VARIANTS:
        opt = orc.make_options(**kw)
        a = animate(MotionChain(spec, W, H, scene, spec.geom_build(scene), *cam, opt), name, scene)
        a.close()
        assert float(a.accum[:, :3].sum()) > 0
        for by_name in (False, True):
            dev = DeviceMotion(rt, by_name)
            b = animate(MotionChain(dev, W, H, scene, dev.geom_build(scene), *cam, opt), name, scene)
            assert same(a.accum, b.accum) and same(a.out, b.out) and same(a.temporal, b.temporal), (kw, by_name)
            for g in dev._geoms:
                g.destroy()
        for reproject in (["surfaces"] if reuse else [True, "surfaces"]):
            for fused in (False, True):
                assert same(_app(rt, c, scene, opt, W, H, cam, name, fused, reproject), a.accum), (kw, fused, reproject)


@pytest.mark.parametrize("math", ["EXACT", "REFERENCE", "FAST"])
def test_identity_in_every_math_mode(rt, c, math):
    """set_triangles with the same vertices before every moved frame (previous triangles byte-equal to the current ones)
    renders what RestirDI renders without it, bit for bit: launch list and fused frame, both reuse weights"""
    name = "lit_blocks_ao"
    make, W, H, cam = SCENES[name]
    W, H = 4 * W, 4 * H
    scene = make()
    rt.set_math_mode(getattr(c, "MATH_" + math))
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    for reuse in (c.REUSE_REFERENCE, c.REUSE_UNBIASED):
        rt.set_reuse_weights(reuse)
        for fused in (False, True):
            a = _app(rt, c, scene, opt, W, H, cam, name, fused, "surfaces", moves=False)
            app = c.RestirDI(rt, W, H, scene, *cam, c.Options.from_numpy(opt), fused=fused, reproject="surfaces")
            for _ in range(2):
                app.frame()
            for eye, center in MOVES[name]:
                app.set_camera(eye, center)
                app.frame()
            b = app.accumulation.to_host().view(np.float32).reshape(-1, 4)
            app.geom.destroy()
            assert same(a, b) and float(a[:, :3].sum()) > 0, (reuse, fused)


def test_overlap_with_prefetch_equals_serial_frames_under_motion(rt, c):
    """frame overlap with the primary-ray prefetch renders what serial frames render while set_triangles refits the tree
    between frames (crt_refit_geometry orders itself after the tail and the prefetch in flight)"""
    name = "cornellbox1"
    make, W, H, cam = SCENES[name]
    W, H = 4 * W, 4 * H
    scene = make()
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    for reuse in (c.REUSE_REFERENCE, c.REUSE_UNBIASED):
        rt.set_reuse_weights(reuse)
        a = _app(rt, c, scene, opt, W, H, cam, name, True, "surfaces")
        b = _app(rt, c, scene, opt, W, H, cam, name, True, "surfaces", overlap=True)
        assert same(a, b) and float(a[:, :3].sum()) > 0, reuse


def test_row_ranges_under_motion(c):
    """three contexts render bands of one image through the motion call (every context reads the whole previous
    Visibility and history, written by all of them) while triangles and camera move twice: equal to one context"""
    name = "cornellbox1"
    scene = small_scene(name)
    W, H, cam = 192, 108, SCENES[name][3]
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    frames = [(cam, scene), (cam, scene)] + [(m, move_triangles(scene, k + 1)) for k, m in enumerate(MOVES[name])]

    def render(bands):
        rts = []
        for y0, y1 in bands:
            r = c.Runtime(0, c.MATH_EXACT)
            r.set_reuse_weights(c.REUSE_UNBIASED)
            r.set_row_range(y0, y1)
            rts.append(r)
        r0 = rts[0]
        n = W * H
        d_t, d_pt = r0.to_device(scene), r0.to_device(scene)
        per = [(r, r.build_geometry(d_t), r.to_device(orc.light_indices(scene))) for r in rts]
        vis, pvis = r0.buffer(c.VISIBILITY, n), r0.buffer(c.VISIBILITY, n)
        b0, b1 = r0.buffer(c.RESERVOIR, n), r0.buffer(c.RESERVOIR, n)
        temporal, acc = r0.buffer(c.RESERVOIR, n).zero(), r0.buffer(c.FLOAT4, n)
        o = c.Options.from_numpy(opt)

        def stage(fn):
            for r, g, d_l in per:
                fn(r, g, d_l)
            for r in rts:
                r.sync()

        prev_rg, cur = None, scene
        for f, ((e, ctr), tris) in enumerate(frames, 1):
            moved = tris is not cur
            if moved:
                d_pt.upload(cur)
                d_t.upload(tris)
                for _, g, _ in per:
                    g.refit()
                cur = tris
            rg, eye = c.lookat(e, ctr, W, H), tuple(float(np.float32(v)) for v in e)
            vis, pvis = pvis, vis
            for r in rts:
                r.clear(acc, W, H)
            stage(lambda r, g, l: r.raycast(W, H, g, d_t, rg, vis))
            stage(lambda r, g, l: r.generate_candidate(W, H, f, g, d_t, vis, eye, l, o, b0))
            if prev_rg is None:
                stage(lambda r, g, l: r.temporal_resampling(W, H, f, g, d_t, vis, eye, o, temporal, b0))
            elif moved:
                stage(lambda r, g, l: r.temporal_resampling_reprojected_motion(W, H, f, g, d_t, vis, eye, o, prev_rg, d_pt,
                                                                               pvis, temporal, b0))
            else:
                stage(lambda r, g, l: r.temporal_resampling_reprojected_surfaces(W, H, f, g, d_t, vis, eye, o, prev_rg,
                                                                                 pvis, temporal, b0))
            prev_rg = rg
            stage(lambda r, g, l: r.save_temporal_reservoir(W, H, b0, temporal))
            bi, bo = b0, b1
            for k in range(int(opt["spatial_resampling_passes"])):
                if k:
                    bi, bo = bo, bi
                stage(lambda r, g, l: r.spatial_resampling(W, H, f, k, g, d_t, vis, eye, o, bi, bo))
            stage(lambda r, g, l: r.resolve(acc, W, H, g, d_t, vis, eye, o, bo))
        out = acc.to_host().view(np.float32).reshape(-1, 4).copy(), bo.to_host().copy(), temporal.to_host().copy()
        for _, g, _ in per:
            g.destroy()
        for r in rts:
            r.close()
        return out

    whole = render([(0, H)])
    bands = render([(0, 37), (37, 71), (71, H)])
    assert all(same(x, y) for x, y in zip(whole, bands))
    assert float(whole[0][:, :3].sum()) > 0


def test_refusals(rt, c):
    tris = lit_blocks_ao()
    cam = ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0))
    W, H, n = 64, 36, 64 * 36
    rt.set_reuse_weights(c.REUSE_UNBIASED)
    d_t, d_pt, d_short = rt.to_device(tris), rt.to_device(tris), rt.to_device(tris[:-1])
    g = rt.build_geometry(d_t)
    rg, eye, o = c.lookat(*cam, W, H), tuple(float(np.float32(v)) for v in cam[0]), c.Options(use_temporal_resampling=1)
    vis, pvis = rt.buffer(c.VISIBILITY, n), rt.buffer(c.VISIBILITY, n)
    prev, res = rt.buffer(c.RESERVOIR, n).zero(), rt.buffer(c.RESERVOIR, n).zero()
    rt.raycast(W, H, g, d_t, rg, vis)
    rt.raycast(W, H, g, d_t, rg, pvis)
    call = rt.temporal_resampling_reprojected_motion
    with pytest.raises(c.CrtError, match="as many triangles"):
        call(W, H, 1, g, d_t, vis, eye, o, rg, d_short, pvis, prev, res)
    with pytest.raises(c.CrtError, match="Visibility must be a buffer of its own"):
        call(W, H, 1, g, d_t, vis, eye, o, rg, d_pt, vis, prev, res)
    with pytest.raises(c.CrtError, match="cannot run in place"):
        call(W, H, 1, g, d_t, vis, eye, o, rg, d_pt, pvis, res, res)
    with pytest.raises(c.CrtError, match="need the previous frame's Visibility"):
        call(W, H, 1, g, d_t, vis, eye, o, rg, d_pt, None, prev, res)
    with pytest.raises(c.CrtError, match="as many triangles"):
        rt.launch("temporal_resampling_reprojected_motion", W, H, 1, g, d_t, vis, c.Float3(*eye), o, rg, d_short, pvis, prev,
                  res)
    null = c._Buffer(None, len(tris) | (1 << 63))
    with pytest.raises(c.CrtError, match="null previous triangle buffer"):
        rt._check(rt.lib.crt_temporal_resampling_reprojected_motion(rt.ctx, W, H, 1, g.handle, d_t.arg(), vis.arg(),
                                                                    c.Float3(*eye), o, rg, null, pvis.arg(), prev.arg(),
                                                                    res.arg()))
    with pytest.raises(c.CrtError, match="null previous triangle buffer"):
        rt._check(rt.lib.crt_restir_set_previous_triangles(rt.ctx, null))
    call(W, H, 1, g, d_t, vis, eye, o, rg, d_pt, pvis, prev, res)  # accepted
    rt.set_reuse_weights(c.REUSE_REFERENCE)
    call(W, H, 1, g, d_t, vis, eye, o, rg, d_pt, None, prev, res)  # the reference's weights do not read it
    g.destroy()
    # the fused frame: the stored array must hold as many triangles
    rt.set_reuse_weights(c.REUSE_UNBIASED)
    app = c.RestirDI(rt, W, H, tris, *cam, c.Options(use_temporal_resampling=1), fused=True)
    app.frame()
    rt.restir_set_previous_frame(rg, pvis)
    rt.restir_set_previous_triangles(d_short)
    with pytest.raises(c.CrtError, match="as many triangles"):
        app.frame()
    rt.restir_set_previous_triangles(d_pt)
    app.frame()  # accepted
    # reprojection stays refused over the direct-store slab links, previous triangles or not
    flags = rt.buffer(np.uint8, 32).zero()
    links = c.SlabLinks()
    links.my_flags = flags.ptr
    rt.slab_set_links(links)
    try:
        with pytest.raises(c.CrtError, match="slab links"):
            app.frame()
    finally:
        rt.slab_set_links(None)
    # a NULL previous camera clears the stored triangles: the short array is not checked any more
    rt.restir_set_previous_triangles(d_short)
    rt.restir_set_previous_frame(None, None)
    app.frame()
    rt.restir_set_previous_frame(rg, pvis)
    app.frame()
    rt.restir_set_previous_frame(None, None)
    app.geom.destroy()
    # RestirDI.set_triangles takes the same number of triangles
    app = c.RestirDI(rt, W, H, tris, *cam, c.Options(use_temporal_resampling=1), fused=True, reproject="surfaces")
    with pytest.raises(ValueError):
        app.set_triangles(tris[:-1])
    app.geom.destroy()


# ---------------------------------------------------------------- row slabs
def _slab_frames(r, scene, name):
    """animate()'s path on a SlabRenderer / SlabGroup / RestirDI: set_triangles and set_camera before each moved frame"""
    for _ in range(2):
        r.frame()
    for k, (eye, center) in enumerate(MOVES[name]):
        r.set_triangles(move_triangles(scene, k + 1))
        r.set_camera(eye, center)
        r.frame()


def test_slab_renderer_follows_motion(c):
    """SlabRenderer(reproject=True | "surfaces").set_triangles renders what RestirDI with set_triangles renders, in fused
    (crt_restir_set_previous_triangles) and drop-in mode (crt_temporal_resampling_reprojected_motion), under both weights
    for "surfaces"; and not what the static assumption renders"""
    import torch

    import slabs

    name = "cornellbox1"
    make, W, H, cam = SCENES[name]
    W, H = 4 * W, 4 * H
    sc = make()
    opt = c.Options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    torch.cuda.set_device(0)
    with torch.cuda.stream(torch.cuda.Stream()):
        for fused in (True, False):
            for rep, reuse in ((True, c.REUSE_REFERENCE), ("surfaces", c.REUSE_REFERENCE), ("surfaces", c.REUSE_UNBIASED)):
                r = slabs.SlabRenderer(torch, None, 0, 1, sc, cam, W, H, fused=fused, reproject=rep)
                r.set_math_mode(c.MATH_EXACT)
                r.set_reuse_weights(reuse)
                _slab_frames(r, sc, name)
                torch.cuda.synchronize()
                got = r.t_acc.cpu().numpy().copy()
                rt = c.Runtime(0, c.MATH_EXACT)
                rt.set_reuse_weights(reuse)
                app = c.RestirDI(rt, W, H, sc, *cam, opt, fused=fused, reproject=rep)
                _slab_frames(app, sc, name)
                want = app.accumulation.to_host().view(np.uint8).reshape(-1)
                assert same(got, want) and want.view(np.float32).sum() > 0, (fused, rep, reuse)
                # the static assumption: the same frames without the previous triangles
                app2 = c.RestirDI(rt, W, H, sc, *cam, opt, fused=fused, reproject=rep)
                for _ in range(2):
                    app2.frame()
                for k, (eye, center) in enumerate(MOVES[name]):
                    app2.triangles.upload(move_triangles(sc, k + 1))
                    app2.geom.refit()
                    app2.set_camera(eye, center)
                    app2.frame()
                assert not same(app2.accumulation.to_host().view(np.uint8).reshape(-1), want), (fused, rep, reuse)
                for a in (app, app2):
                    a.geom.destroy()
                rt.close()


def test_slab_group_equals_one_slab_under_motion(c):
    """three slabs of 960x540 on one GPU linked by plain pointers, unbiased weights, triangles and camera moving twice
    (SlabGroup.set_triangles: the shared scene array rewritten and the shared tree refitted once the slabs' frames are
    done): equal to one slab bit for bit"""
    import torch

    import slabs

    name = "lit_blocks_ao"
    sc = SCENES[name][0]()
    W, H, cam = 960, 540, SCENES[name][3]
    torch.cuda.set_device(0)
    with torch.cuda.stream(torch.cuda.Stream()):
        part = slabs.SlabGroup(torch, None, 0, 1, sc, cam, W, H, sub=3)
        full = slabs.SlabRenderer(torch, None, 0, 1, sc, cam, W, H, fused=True)
        for r in (part, full):
            r.set_reuse_weights(c.REUSE_UNBIASED)
            _slab_frames(r, sc, name)
        part.join()
        torch.cuda.synchronize()
        part.check()
        assert part.p2p and len(part.slabs) == 3
        for sl in part.slabs:
            for tname, elem in (("t_acc", 16), ("t_pix", 4), ("t_vis", 16)):
                a = sl._rows(getattr(sl, tname), elem, sl.y0, sl.y1)
                b = full._rows(getattr(full, tname), elem, sl.y0, sl.y1)
                assert torch.equal(a, b), (tname, sl.rank)
        assert float(full.t_acc.view(torch.float32).sum()) > 0
        part.close()


# ---------------------------------------------------------------- unbiasedness
STEP = np.array([1.2, 0.6, -0.8])  # per frame; the chains' four eyes end at CAM_RIDGES


def flipped(tris):
    """the ridged floor with peaks and valleys swapped: each face's tilt towards the light reverses (the light stays)"""
    out = tris.copy()
    y = out["vertices"][:-2, :, 1]
    out["vertices"][:-2, :, 1] = y.max() - y
    return out


def _animated_chains(rt, c, tris, mode, N, arm, W=128, H=96):
    """N independent chains of 4 frames (history zeroed, disjoint frame numbers, temporal + 3 spatial passes, no
    accumulation): the floor flips before every frame and ends as `tris`, the camera steps towards CAM_RIDGES.  arm:
    "motion" (RestirDI(reproject="surfaces").set_triangles), "static" (the same look-ups without the previous triangles:
    the vertices are written and the tree refitted behind RestirDI's back), "none" (no reprojection); the lit faces'
    region mean of each chain's last frame"""
    rt.set_reuse_weights(mode)
    opt = c.Options(accumulate=0, use_temporal_resampling=1, use_spatial_resampling=1)
    eye0, center = np.array(CAM_RIDGES[0]), CAM_RIDGES[1]
    app = c.RestirDI(rt, W, H, tris, *CAM_RIDGES, opt, fused=True, reproject="surfaces" if arm != "none" else False)
    states = [tris, flipped(tris)]
    means = []
    for _ in range(N):
        app.temporal.zero()
        app.prev_raygen = None
        for k in (3, 2, 1, 0):
            t = states[k % 2]
            if arm == "motion":
                app.set_triangles(t)
            else:
                app.triangles.upload(t)
                app.geom.refit()
            app.set_camera(tuple(eye0 + k * STEP), center)
            app.frame()
        means.append(app.accumulation.to_host().view(np.float32).reshape(-1, 4)[:, :3].astype(np.float64))
    app.geom.destroy()
    return means


def test_unbiased_motion_reuse_matches_plain_ris(rt, c):
    """the point of the feature.  The ridged floor's sawtooth flips every frame, so a face lit this frame was tilted away
    from the light last frame; 96 chains of 4 frames against 96 frames of plain RIS on the final geometry at the final
    view, region means over the lit faces, z-score of the difference from the across-chain variance.  Bar: unbiased
    weights with motion z < 4.  The motion-unaware arms (reproject="surfaces" without the previous triangles, and no
    reprojection) are reported, not barred: the reference's target function takes absolute cosines, so p_hat_h(y) > 0 on
    either tilt and Z counts the history whatever surface S_h is rebuilt on; a wrong S_h only changes c_h, which 1/Z
    weights tolerate (DESIGN.md section 17, "What the test can see").  Measured on a B200 (1000 W power limit), N = 96:
    motion z = 0.02, static z = 0.14, no reprojection z = 0.30."""
    rt.set_math_mode(c.MATH_REFERENCE)
    tris = ridged_floor()
    N = 96
    ris, lit = _last_frames(rt, c, tris, False, c.REUSE_REFERENCE, N)
    assert 0.3 < lit.mean() < 0.7 and ris.mean() > 0
    z, rel = {}, {}
    for arm in ("motion", "static", "none"):
        m = np.array([a[lit].sum(1).mean() for a in _animated_chains(rt, c, tris, c.REUSE_UNBIASED, N, arm)])
        z[arm] = abs(m.mean() - ris.mean()) / np.sqrt(m.var(ddof=1) / N + ris.var(ddof=1) / N)
        rel[arm] = m.mean() / ris.mean() - 1.0
    print("ridged floor flipping every frame, unbiased weights: " +
          ", ".join("%s z = %.2f (%+.4f)" % (k, z[k], rel[k]) for k in z))
    assert z["motion"] < 4
