"""Unbiased reuse weights on row slabs (crt_restir_set_halo_surfaces) on the GPU: contexts that render bands of one image
in the fused frame — their halo rows exchanged between stages, as slabs.exchange does — equal one whole-image context bit
for bit in every math mode, with uniform and power light selection and a moving camera, also with reprojection onto the
previous frame's surfaces; the halo G-buffer records equal the owners'; slabs.SlabGroup over direct-store links equals one
slab; the opt-in changes nothing under the reference's weights; the new refusal."""
import os
import subprocess
import sys

import numpy as np
import pytest

import orc
from helpers import same, scene, small_scene
from test_reuse_reprojection import MOVES
from test_reuse_weights import SCENES

pytestmark = pytest.mark.gpu

CAM_RESTIR = ((-0.579885, 22.194597, -6.567105), (5.224952, 20.847435, 1.431192))  # 10_restir_di.cpp:188-189
POISON = 0xAB
THIN = [(0, 37), (37, 53), (53, 144)]  # edges on no multiple of 8; the middle band is thinner than the halo


def _import():
    import torch

    import cedecrt
    import slabs

    return torch, cedecrt, slabs


class Band:
    """one context on rows [y0, y1) with full-size buffers of its own (torch tensors), rows outside its range poisoned"""

    def __init__(self, torch, c, tris, W, H, y0, y1, math, lights, halo=True, reuse=None):
        self.torch, self.c, self.W, self.H, self.y0, self.y1 = torch, c, W, H, y0, y1
        n = W * H
        self.rt = c.Runtime(0, math)
        self.rt.set_reuse_weights(c.REUSE_UNBIASED if reuse is None else reuse)
        self.rt.set_light_sampling(lights)
        self.rt.set_row_range(y0, y1)
        if halo:
            self.rt.restir_set_halo_surfaces(True)
        dev = torch.device("cuda", 0)
        self.d_tris = self.rt.to_device(tris)
        self.d_lights = self.rt.to_device(orc.light_indices(tris))
        self.geom = self.rt.build_geometry(self.d_tris)
        sizes = {"pix": 4, "acc": 16, "vis": 16, "vis_prev": 16, "r0": 76, "r1": 76, "tmp": 76}
        self.t = {k: torch.full((e * n,), POISON, dtype=torch.uint8, device=dev) for k, e in sizes.items()}
        self.zero_own("acc", 16)
        self.zero_own("tmp", 76)  # no history; the SoA records of the own rows sit in every plane
        self.prev_rg = None

    def rows(self, name, elem, a, b):
        return self.t[name][(self.H - b) * self.W * elem:(self.H - a) * self.W * elem]

    def zero_own(self, name, elem):
        if name == "tmp":  # SoA: planes of 32, 32 and 8 bytes per pixel over W * H pixels
            import slabs

            for s0, s1 in slabs.row_byte_ranges(self.W, self.H, (self.y0, self.y1), slabs.SOA_RESERVOIR):
                self.t[name][s0:s1] = 0
        else:
            self.rows(name, elem, self.y0, self.y1).zero_()

    def bufs(self):
        c, n, w = self.c, self.W * self.H, self.rt.wrap
        b = {k: w(v.data_ptr(), dt, cnt) for k, (v, dt, cnt) in {
            "pix": (self.t["pix"], np.uint8, 4 * n), "acc": (self.t["acc"], c.FLOAT4, n), "vis": (self.t["vis"], c.VISIBILITY, n),
            "r0": (self.t["r0"], c.RESERVOIR, n), "r1": (self.t["r1"], c.RESERVOIR, n), "tmp": (self.t["tmp"], c.RESERVOIR, n)}.items()}
        self._keep = b
        return self.rt.restir_buffers(b["pix"], b["acc"], b["vis"], b["r0"], b["r1"], b["tmp"])

    def prev_vis_buffer(self):
        self._keep_prev = self.rt.wrap(self.t["vis_prev"].data_ptr(), self.c.VISIBILITY, self.W * self.H)
        return self._keep_prev

    def final_reservoirs(self, o):
        """the frame's final reservoirs (crt_restir_output_buffer) in AoS"""
        k = "tmp" if not o.use_spatial_resampling or o.spatial_resampling_passes <= 0 else (
            "r1" if o.spatial_resampling_passes % 2 else "r0")
        n = self.W * self.H
        src = self.rt.wrap(self.t[k].data_ptr(), self.c.RESERVOIR, n)
        out = self.rt.buffer(self.c.RESERVOIR, n)
        self.rt.reservoir_export_aos(self.W, self.H, src, out)
        return out.to_host()

    def gbuf(self):
        """the context's G-buffer (g0: 16 B/px, g1: 8 B/px) as numpy"""
        import slabs

        n = self.W * self.H
        base = self.rt.restir_reserve(self.W, self.H)
        self.rt.sync()
        t = self.torch.as_tensor(slabs.CudaArrayView(base, 24 * n), device="cuda").cpu().numpy()
        return t[:16 * n].reshape(n, 16), t[16 * n:24 * n].reshape(n, 8)

    def close(self):
        self.geom.destroy()
        self.rt.close()


def render(torch, c, slabs, tris, W, H, bands, math, lights, o, cams, reproject=False, halo=True, reuse=None):
    """the fused frame on each band (crt_restir_frame_begin / spatial_pass / frame_end), the camera of frame f = cams[f - 1]
    (set_camera semantics: the accumulation of the own rows cleared on a move).  Before spatial pass k every band receives
    the rows of pass k's input within its halo from their owners; with reprojection, before every frame after the first,
    every row of `temporal` and of last frame's Visibility."""
    B = [Band(torch, c, tris, W, H, y0, y1, math, lights, halo, reuse) for y0, y1 in bands]
    h = slabs.halo_rows(o.spatial_resampling_radius)

    def sync():
        for b in B:
            b.rt.sync()
        torch.cuda.synchronize()

    def gather(name, layout, reach):
        for b in B:
            for a in B:
                if a is b:
                    continue
                lo, hi = max(a.y0, b.y0 - reach), min(a.y1, b.y1 + reach)
                if lo < hi:
                    for s0, s1 in slabs.row_byte_ranges(W, H, (lo, hi), layout):
                        b.t[name][s0:s1].copy_(a.t[name][s0:s1])
        torch.cuda.synchronize()

    prev = None
    for f, (e, ctr) in enumerate(cams, 1):
        rg, eye = c.lookat(e, ctr, W, H), tuple(float(np.float32(v)) for v in e)
        if prev is not None and prev != (e, ctr):
            for b in B:
                b.zero_own("acc", 16)
        if reproject:
            for b in B:
                b.t["vis"], b.t["vis_prev"] = b.t["vis_prev"], b.t["vis"]
            if f > 1:
                gather("tmp", slabs.SOA_RESERVOIR, H)
                gather("vis_prev", slabs.AOS_VISIBILITY, H)
        bufs = [b.bufs() for b in B]
        for b, bf in zip(B, bufs):
            if reproject:
                b.rt.restir_set_previous_frame(b.prev_rg, b.prev_vis_buffer())
            b.rt.restir_frame_begin(W, H, f, b.geom, b.d_tris, rg, eye, b.d_lights, o, bf)
            b.prev_rg = rg
        sync()
        for k in range(o.spatial_resampling_passes if o.use_spatial_resampling else 0):
            gather("tmp" if k == 0 else ("r1" if k % 2 else "r0"), slabs.SOA_RESERVOIR, h)
            for b, bf in zip(B, bufs):
                b.rt.restir_spatial_pass(W, H, f, k, b.geom, b.d_tris, eye, o, bf)
            sync()
        for b, bf in zip(B, bufs):
            b.rt.restir_frame_end(W, H, b.geom, b.d_tris, eye, o, bf)
        sync()
        prev = (e, ctr)
    for b in B:
        if reproject:
            b.rt.restir_set_previous_frame(None, None)
    return B, h


def _opts(c, radius=30.0):
    return c.Options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1, spatial_resampling_radius=radius)


def _check_bands(torch, slabs, whole, B, h, o, H, reproject=False):
    """own rows equal the whole-image context; rows nobody gave the band stay poisoned"""
    w = whole[0]
    fin_w = w.final_reservoirs(o)
    for b in B:
        for name, elem in (("acc", 16), ("pix", 4), ("vis", 16)):
            assert torch.equal(b.rows(name, elem, b.y0, b.y1), w.rows(name, elem, b.y0, b.y1)), (name, b.y0, b.y1)
        fin = b.final_reservoirs(o)
        own = slice((H - b.y1) * b.W, (H - b.y0) * b.W)
        assert same(fin[own], fin_w[own]), ("reservoirs", b.y0, b.y1)
        # the library writes the host's buffers in the band's own rows only
        outside = [(0, b.y0), (b.y1, H)]
        for a, z in outside:
            if a >= z:
                continue
            for name, elem in (("acc", 16), ("pix", 4)) + ((("vis", 16),) if not reproject else ()):
                assert bool((b.rows(name, elem, a, z) == POISON).all()), (name, a, z)
        if not reproject:  # reservoir rows beyond the halo: nobody gave them to the band
            for a, z in ((0, max(0, b.y0 - h)), (min(H, b.y1 + h), H)):
                if a < z:
                    for name in ("r0", "r1", "tmp"):
                        for s0, s1 in slabs.row_byte_ranges(b.W, H, (a, z), slabs.SOA_RESERVOIR):
                            assert bool((b.t[name][s0:s1] == POISON).all()), (name, a, z)
        # the halo G-buffer records are the owner's (the whole-image context's), bit for bit, for diffuse pixels
        g0b, g1b = b.gbuf()
        g0w, g1w = w.gbuf()
        for a, z in ((max(0, b.y0 - h), b.y0), (b.y1, min(H, b.y1 + h))):
            if a >= z:
                continue
            sl = slice((H - z) * b.W, (H - a) * b.W)
            d = w.diffuse[sl]
            assert (g0b[sl][d] == g0w[sl][d]).all() and (g1b[sl][d] == g1w[sl][d]).all(), ("halo records", a, z)


def _diffuse_of(band, tris):
    idx = band.t["vis"].cpu().numpy().view(orc.VISIBILITY)["index"]
    d = idx >= 0
    em = (tris["emissive"] > 0).any(1)
    d[d] = ~em[idx[d]]
    return d


def _run(name, math_name, lights_name, radius=30.0, bands=THIN, reproject=False):
    torch, c, slabs = _import()
    make, W, H, cam = SCENES[name]
    W, H = 4 * W, 4 * H
    tris = make()
    math = {"exact": c.MATH_EXACT, "reference": c.MATH_REFERENCE, "fast": c.MATH_FAST}[math_name]
    lights = c.LIGHTS_POWER if lights_name == "power" else c.LIGHTS_UNIFORM
    o = _opts(c, radius)
    cams = [cam, cam] + MOVES[name]
    whole, _ = render(torch, c, slabs, tris, W, H, [(0, H)], math, lights, o, cams, reproject)
    whole[0].diffuse = _diffuse_of(whole[0], tris)
    B, h = render(torch, c, slabs, tris, W, H, bands, math, lights, o, cams, reproject)
    try:
        assert float(whole[0].rows("acc", 16, 0, H).view(torch.float32).sum()) > 0
        _check_bands(torch, slabs, whole, B, h, o, H, reproject)
    finally:
        for b in B + whole:
            b.close()


@pytest.mark.parametrize("lights", ["uniform", "power"])
@pytest.mark.parametrize("math", ["exact", "reference", "fast"])
@pytest.mark.parametrize("name", ["cornellbox1", "lit_blocks_ao"])
def test_bands_equal_one_context(name, math, lights):
    """three bands (one thinner than the halo, so rows come from a band that is not adjacent), 4 frames with a camera that
    moves twice: accumulation, pixels, Visibility and final reservoirs of each band's rows equal one whole-image context
    bit for bit; the halo G-buffer records equal the owner's; rows outside the band stay untouched"""
    _run(name, math, lights)


def test_bands_at_a_larger_radius():
    """spatial_resampling_radius 45: the halo reaches halo_rows(45) > 87 rows"""
    _, _, slabs = _import()
    assert slabs.halo_rows(45.0) > 87
    _run("cornellbox1", "exact", "uniform", radius=45.0, bands=[(0, 61), (61, 101), (101, 144)])


@pytest.mark.parametrize("math", ["exact", "reference"])
@pytest.mark.parametrize("lights", ["uniform", "power"])
def test_bands_with_reprojection(math, lights):
    """as above with crt_restir_set_previous_frame: before every frame after the first each band receives every row of
    `temporal` and of last frame's Visibility; the camera moves twice"""
    _run("cornellbox1", math, lights, reproject=True)


def _group_vs_one(overlap):
    torch, c, slabs = _import()
    tris = scene("blocks_restir")
    W, H = 960, 540
    e, ctr = np.asarray(CAM_RESTIR[0]), np.asarray(CAM_RESTIR[1])
    move = (tuple(e + (0.4, -0.2, 0.1)), tuple(ctr + (0.1, 0.0, -0.1)))
    torch.cuda.set_device(0)
    with torch.cuda.stream(torch.cuda.Stream()):
        part = slabs.SlabGroup(torch, None, 0, 1, tris, CAM_RESTIR, W, H, sub=3, overlap=overlap)
        full = slabs.SlabRenderer(torch, None, 0, 1, tris, CAM_RESTIR, W, H, fused=True)
        for r in (part, full):
            r.set_reuse_weights(c.REUSE_UNBIASED)
        for k in range(4):
            if k == 2:
                part.set_camera(*move)
                full.set_camera(*move)
            part.frame()
            full.frame()
        part.join()
        torch.cuda.synchronize()
        part.check()
        assert part.p2p and len(part.slabs) == 3
        for sl in part.slabs:
            for name, elem in (("t_acc", 16), ("t_pix", 4), ("t_vis", 16)):
                a = sl._rows(getattr(sl, name), elem, sl.y0, sl.y1)
                b = full._rows(getattr(full, name), elem, sl.y0, sl.y1)
                assert torch.equal(a, b), (name, sl.rank)
        part.close()


def test_slab_group_unbiased_on_one_gpu():
    """three slabs of 960x540 on one GPU linked by plain pointers (direct halo stores), unbiased weights, 4 frames with a
    camera move: equal to one slab bit for bit"""
    _group_vs_one(False)


def test_slab_group_unbiased_with_frame_overlap():
    _group_vs_one(True)


def test_halo_surfaces_change_nothing_under_reference_weights():
    """the opt-in on a band under the reference's weights, and on the whole image under unbiased ones: the same launches and
    the same bits as without it"""
    torch, c, slabs = _import()
    make, W, H, cam = SCENES["lit_blocks_ao"]
    W, H = 4 * W, 4 * H
    tris = make()
    o = _opts(c)
    cams = [cam, cam] + MOVES["lit_blocks_ao"]
    for bands, reuse in (([(37, 101)], c.REUSE_REFERENCE), ([(0, H)], c.REUSE_UNBIASED)):
        runs = []
        for halo in (False, True):
            B, _ = render(torch, c, slabs, tris, W, H, bands, c.MATH_REFERENCE, c.LIGHTS_UNIFORM, o, cams, halo=halo, reuse=reuse)
            b = B[0]
            runs.append((b.rt.launch_count(), b.rows("acc", 16, b.y0, b.y1).clone(), b.final_reservoirs(o)))
            b.close()
        assert runs[0][0] == runs[1][0], (bands, runs[0][0], runs[1][0])
        assert torch.equal(runs[0][1], runs[1][1]) and same(runs[0][2], runs[1][2])


def test_slab_renderer_surfaces_equals_reproject_under_reference_weights():
    """SlabRenderer(reproject="surfaces") under the reference's weights renders what reproject=True renders (fused and
    drop-in), and under unbiased weights what cedecrt.RestirDI(reproject="surfaces") renders"""
    torch, c, slabs = _import()
    make, W, H, cam = SCENES["cornellbox1"]
    W, H = 4 * W, 4 * H
    tris = make()
    torch.cuda.set_device(0)
    with torch.cuda.stream(torch.cuda.Stream()):
        for fused in (True, False):
            out = {}
            for rep, reuse in ((True, c.REUSE_REFERENCE), ("surfaces", c.REUSE_REFERENCE), ("surfaces", c.REUSE_UNBIASED)):
                r = slabs.SlabRenderer(torch, None, 0, 1, tris, cam, W, H, fused=fused, reproject=rep)
                r.set_math_mode(c.MATH_EXACT)
                r.set_reuse_weights(reuse)
                for k in range(4):
                    if k >= 2:
                        r.set_camera(*MOVES["cornellbox1"][k - 2])
                    r.frame()
                torch.cuda.synchronize()
                out[(rep, reuse)] = r.t_acc.cpu().numpy().copy()
            assert same(out[(True, c.REUSE_REFERENCE)], out[("surfaces", c.REUSE_REFERENCE)]), fused
            rt = c.Runtime(0, c.MATH_EXACT)
            rt.set_reuse_weights(c.REUSE_UNBIASED)
            app = c.RestirDI(rt, W, H, tris, *cam, c.Options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1),
                             fused=fused, reproject="surfaces")
            for k in range(4):
                if k >= 2:
                    app.set_camera(*MOVES["cornellbox1"][k - 2])
                app.frame()
            acc = app.accumulation.to_host().view(np.uint8).reshape(-1)
            assert same(acc, out[("surfaces", c.REUSE_UNBIASED)]), fused
            assert not same(out[("surfaces", c.REUSE_UNBIASED)], out[("surfaces", c.REUSE_REFERENCE)])
            app.geom.destroy()
            rt.close()


def test_refusal_of_a_radius_beyond_the_halo():
    """crt_restir_spatial_pass with a radius that reaches further than the rows crt_restir_frame_begin covered"""
    torch, c, slabs = _import()
    tris = small_scene("cornellbox1")
    W, H = 256, 144
    cam = SCENES["cornellbox1"][3]
    b = Band(torch, c, tris, W, H, 37, 101, c.MATH_EXACT, c.LIGHTS_UNIFORM)
    try:
        bufs = b.bufs()
        rg, eye = c.lookat(*cam, W, H), tuple(float(np.float32(v)) for v in cam[0])
        o30, o45 = _opts(c, 30.0), _opts(c, 45.0)
        b.rt.restir_frame_begin(W, H, 1, b.geom, b.d_tris, rg, eye, b.d_lights, o30, bufs)
        with pytest.raises(c.CrtError, match="do not reach"):
            b.rt.restir_spatial_pass(W, H, 1, 0, b.geom, b.d_tris, eye, o45, bufs)
        b.rt.restir_spatial_pass(W, H, 1, 0, b.geom, b.d_tris, eye, o30, bufs)  # accepted
        b.rt.restir_frame_begin(W, H, 2, b.geom, b.d_tris, rg, eye, b.d_lights, o45, bufs)
        b.rt.restir_spatial_pass(W, H, 2, 0, b.geom, b.d_tris, eye, o30, bufs)  # a shorter reach is covered
        # without the opt-in the row range stays refused, with the message it always had
        b.rt.restir_set_halo_surfaces(False)
        with pytest.raises(c.CrtError, match="whole image"):
            b.rt.restir_frame_begin(W, H, 3, b.geom, b.d_tris, rg, eye, b.d_lights, o30, bufs)
        b.rt.sync()
    finally:
        b.close()


@pytest.mark.parametrize("mode", ["fused", "fused_nccl", "group", "fused_reproject_surfaces", "dropin_reproject_surfaces"])
def test_unbiased_slabs_on_gpus(mode):
    """N row slabs on N GPUs under unbiased weights (tests/gpu_slab_reuse_worker.py) reproduce one slab bit for bit on their
    rows (needs >= 2 GPUs)"""
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 4 if n >= 4 else 2
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                        "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 200),
                        os.path.join(root, "tests", "gpu_slab_reuse_worker.py")], env=dict(os.environ, SLAB_MODE=mode),
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "GPU_SLABS_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])
    if mode in ("fused", "group"):
        assert "p2p True" in r.stdout, r.stdout[-500:]
