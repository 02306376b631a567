"""Shared helpers for the test-suite (test infrastructure)."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RES_FIELDS = ("origin_position", "origin_normal", "hit_position", "hit_normal", "radiance", "visibility", "w_sum",
              "ucw", "M")


def golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def small_scene(name):
    return np.ascontiguousarray(golden("scenes_small.npz")[name])


# blocks_pt (852 070 triangles, 4 lights) and blocks_restir (1 598 368 triangles, 145 982 lights) are tens of MB: the
# repository does not hold them, so a seeded procedural city of the same size and character stands in for each
STAND_INS = {"blocks_pt": dict(n_blocks=71006, seed=8, extent=200.0, emissive_fraction=5e-5),
             "blocks_restir": dict(n_blocks=133197, seed=10, extent=400.0, emissive_fraction=0.0913)}


def scene(name):
    """a scene the examples load, from the repository alone: cornellbox1 and blocks_ao as the reference loader produced
    them (golden/scenes_small.npz), blocks_pt and blocks_restir as their procedural stand-ins (STAND_INS)"""
    if name in STAND_INS:
        import scenes

        return scenes.procedural_blocks(**STAND_INS[name])
    return small_scene(name)


def same(a, b):
    """bit-level equality that treats NaN == NaN (compares raw bytes of float arrays)."""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def reservoir_mismatch(a, b):
    """number of pixels whose reservoirs differ in any field (padding bytes ignored)."""
    if len(a) == 0:
        return 0
    bad = np.zeros(len(a), bool)
    for f in RES_FIELDS:
        x, y = a[f], b[f]
        if x.dtype.kind == "f":
            x, y = x.view(np.uint32), y.view(np.uint32)
        d = x != y
        bad |= d.reshape(len(a), -1).any(1)
    return int(bad.sum())


class DeviceAsOracle:
    """Adapter: drives libcedecrt through its C ABI with the call shapes of oracle/orc.py:Oracle, so the same
    numpy-level drivers (orc.RestirChain) run the CUDA path.  Inputs are uploaded and outputs downloaded on
    every call — this is a test harness, not the product's frame loop (cedecrt.RestirDI keeps buffers resident)."""

    kind = "cuda"

    def __init__(self, rt):
        import cedecrt

        self.rt, self.c = rt, cedecrt
        self._geoms = []

    def set_math_mode(self, m):
        self.rt.set_math_mode(m)

    def geom_build(self, tris):
        d_tris = self.rt.to_device(tris)
        g = self.rt.build_geometry(d_tris)
        self._geoms.append(g)
        return g

    def geom_free(self, g):
        g.destroy()

    def lookat(self, eye, center, W, H):
        return self.c.lookat(eye, center, W, H)

    def _opt(self, opt):
        return opt if isinstance(opt, self.c.Options) else self.c.Options.from_numpy(opt)

    def _rg(self, rg):
        if isinstance(rg, self.c.RayGenerator):
            return rg
        out = self.c.RayGenerator()
        import ctypes as C

        C.memmove(C.byref(out), rg.tobytes(), 36)
        return out

    def raycast(self, W, H, g, tris, rg, vis=None):
        d = self.rt.buffer(self.c.VISIBILITY, W * H)
        self.rt.raycast(W, H, g, g.triangles, self._rg(rg), d)
        out = d.to_host()
        if vis is not None:
            vis[:] = out
            return vis
        return out

    def generate_candidate(self, W, H, frame, g, tris, vis, eye, lights, opt, res=None):
        d_v, d_l = self.rt.to_device(vis), self.rt.to_device(lights)
        d_r = self.rt.buffer(self.c.RESERVOIR, W * H)
        self.rt.generate_candidate(W, H, frame, g, g.triangles, d_v, tuple(eye), d_l, self._opt(opt), d_r)
        out = d_r.to_host()
        if res is not None:
            res[:] = out
            return res
        return out

    def temporal_resampling(self, W, H, frame, g, tris, vis, eye, opt, prev, res):
        d_v, d_p, d_r = self.rt.to_device(vis), self.rt.to_device(prev), self.rt.to_device(res)
        self.rt.temporal_resampling(W, H, frame, g, g.triangles, d_v, tuple(eye), self._opt(opt), d_p, d_r)
        res[:] = d_r.to_host()
        return res

    def temporal_resampling_reprojected(self, W, H, frame, g, tris, vis, eye, opt, prev_rg, prev, res):
        d_v, d_p, d_r = self.rt.to_device(vis), self.rt.to_device(prev), self.rt.to_device(res)
        self.rt.temporal_resampling_reprojected(W, H, frame, g, g.triangles, d_v, tuple(eye), self._opt(opt), self._rg(prev_rg),
                                                d_p, d_r)
        res[:] = d_r.to_host()
        return res

    def save_temporal_reservoir(self, W, H, src, dst):
        d_s, d_d = self.rt.to_device(src), self.rt.to_device(dst)
        self.rt.save_temporal_reservoir(W, H, d_s, d_d)
        dst[:] = d_d.to_host()
        return dst

    def spatial_resampling(self, W, H, frame, pas, g, tris, vis, eye, opt, rin, rout):
        d_v, d_i, d_o = self.rt.to_device(vis), self.rt.to_device(rin), self.rt.to_device(rout)
        self.rt.spatial_resampling(W, H, frame, pas, g, g.triangles, d_v, tuple(eye), self._opt(opt), d_i, d_o)
        rout[:] = d_o.to_host()
        return rout

    def resolve(self, accum, W, H, g, tris, vis, eye, opt, res):
        d_a = self.rt.to_device(np.ascontiguousarray(accum, np.float32).reshape(-1))
        d_a.dtype, d_a.n = self.c.FLOAT4, W * H
        d_v, d_r = self.rt.to_device(vis), self.rt.to_device(res)
        self.rt.resolve(d_a, W, H, g, g.triangles, d_v, tuple(eye), self._opt(opt), d_r)
        accum[:] = d_a.to_host().view(np.float32).reshape(accum.shape)
        return accum

    def tone_mapping(self, accum, W, H, pixels=None):
        d_a = self.rt.to_device(np.ascontiguousarray(accum, np.float32).reshape(-1))
        d_a.dtype, d_a.n = self.c.FLOAT4, W * H
        d_p = self.rt.buffer(np.uint8, 4 * W * H)
        self.rt.tone_mapping(d_p, d_a, W, H)
        return d_p.to_host()

    def path_trace(self, example, W, H, frame, g, tris, lights, rg, opt, accum):
        d_a = self.rt.to_device(np.ascontiguousarray(accum, np.float32).reshape(-1))
        d_a.dtype, d_a.n = self.c.FLOAT4, W * H
        d_l = self.rt.to_device(lights if len(lights) else np.zeros(1, np.uint32))
        d_l.n = len(lights)
        self.rt.path_trace(example, W, H, frame, g, g.triangles, d_l, self._rg(rg), self._opt(opt), d_a)
        accum[:] = d_a.to_host().view(np.float32).reshape(accum.shape)
        return accum

    def ao(self, W, H, g, tris, rg, n_rays=64):
        d_p = self.rt.buffer(np.uint8, 4 * W * H)
        self.rt.ao(d_p, self._rg(rg), W, H, g, g.triangles, n_rays)
        return d_p.to_host()
