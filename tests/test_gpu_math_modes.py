"""The contracted-arithmetic builds of the fused frame, stage by stage, against the CPU oracle.

CRT_MATH_REFERENCE (the context's default: kernels_fast.cu built with FMA contraction) and CRT_MATH_FAST (built with
-use_fast_math) change the bits of every float result, so they cannot be tested bit for bit.  test_gpu_parity.py checks
them only through the mean relative L1 of a 64-frame image, which a bug confined to these builds can pass by moving a
few percent of pixels by a few percent.  Here each stage of the fused frame runs in every math mode from the oracle's
own input state (oracle/port in exact arithmetic, imported with crt_reservoir_import_aos) and its output is compared
with the oracle's output of the same stage on the same input:

  frame_begin   primary rays (exact in every mode: bit-exact), RIS candidates + temporal merge
  spatial k     one crt_restir_spatial_pass per pass
  frame_end     resolve into the accumulation, then tone mapping

An ulp of difference may flip a RIS or merge decision, so each diffuse pixel is either *same* (equal M, equal
visibility, a selected sample at the oracle's hit position to within 1e-4 relative) or *flipped*; flipped pixels whose
M alone differs, by one, are told apart from the others.  Bars: both fractions of flipped pixels per stage, and the
relative error of w_sum, ucw and radiance of the same pixels (99.9th percentile and mean), and of the radiance resolve
adds to them.  Sky and emissive pixels carry no reservoir work and stay bit-exact.  EXACT mode runs through the same harness
and must be bit-exact everywhere, which shows the harness itself feeds both sides the same state.

Independent of the oracle, every output reservoir satisfies the invariant its last step establishes (ucw_of,
restir_core.cuh; 10_restir_di.cu temporal/spatial resampling): ucw = w_sum / (M * p_hat), p_hat the target function of
the stored sample *at this pixel's surface* — the pixel's point and normal, not the sample's origin fields, which after
a spatial merge are the neighbour's.  It is recomputed here in float64 from the reservoir's hit position, hit normal and
radiance and the pixel's primitive and barycentrics, for the oracle and for the device.

Measured on an NVIDIA B200 (1000 W power limit); the numbers are in each bar's comment and in DESIGN.md section 2.
"""
import numpy as np
import pytest

import cedecrt
import orc
from helpers import reservoir_mismatch, same, scene, small_scene

pytestmark = pytest.mark.gpu

CAM_AO = ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0))
CAM_RESTIR = ((-0.579885, 22.194597, -6.567105), (5.224952, 20.847435, 1.431192))  # 10_restir_di.cpp:188-189
CAM_BUMPS = ((0.0, 7.0, 11.0), (0.0, 0.0, 0.0))
KW = dict(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
MODES = {"exact": cedecrt.MATH_EXACT, "reference": cedecrt.MATH_REFERENCE, "libdevice": cedecrt.MATH_LIBDEVICE,
         "fast": cedecrt.MATH_FAST}
K_SKIP = 0x20000000  # restir_fast.cuh: kSkipBit in word 6 of plane 0 (the flags | M word)

# Bars per mode, from the largest value measured over the four scenes on an NVIDIA B200 (1000 W power limit), with a margin
# of 1.5-4x (measured value in brackets):
#   m1_begin / m1_spatial  fraction of diffuse pixels that differ in M alone, by one (same sample, same visibility), after
#                          frame_begin / after a spatial pass
#   other                  fraction of diffuse pixels with any other difference: another sample, another visibility, M
#                          off by more than one — at every stage
#   rel999 / rel_mean      99.9th percentile and mean of the relative error of w_sum, ucw, radiance of the same pixels
#   inv_frac / inv_med     fraction of reservoirs off the float64 invariant by more than 1e-3, median deviation
#   res_rel999 / _mean     resolve: the same statistics of the radiance it adds, for pixels whose final reservoirs decided
#                          alike (those whose resolve ray grazes differently, off by more than 1e-3, count against m1_spatial)
# Why M alone differs by one: the temporal merge keeps trunc(M * w), w = pow(cos(n_pixel, n_history), 8) * ..., and the cosine
# of a float normal with itself is often an ulp below 1.  That is the reference's own behaviour: in a run of one mode on its
# own history (blocks_ao 320x180, frames 2-6), the temporal M of 9.6 % of the diffuse pixels falls one below 32 f in EXACT
# (the oracle's arithmetic) and LIBDEVICE, 13.4 % in REFERENCE, 5.2 % in FAST; on the heightfield 35 %, 35 %, 36 %, 11 %.
# Which pixels lose one depends on the last bits of their normals, so a history from the oracle merged with this mode's
# normals moves some pixels across.  LIBDEVICE's candidate stage is uncontracted: no flip there; its spatial flips come
# from libdevice's log / sincos in the neighbour offsets.
BARS = {
    "reference": dict(m1_begin=0.15,      # [8.7e-2, heightfield; 0 on the stand-in]
                      m1_spatial=5e-3,    # [2.7e-3, blocks_restir band]
                      other=2e-4,         # [5.4e-5 (2 pixels), heightfield, frame_begin]
                      rel999=3e-5,        # [1.2e-5]
                      rel_mean=1e-6,      # [2.1e-7]
                      inv_frac=1e-3,      # [0]
                      inv_med=4e-7,       # [1.5e-7; the oracle itself: 1.6e-7]
                      res_rel999=3e-5,    # [1.2e-5]
                      res_rel_mean=1e-6),  # [1.9e-7]
    "libdevice": dict(m1_begin=1e-3, m1_spatial=5e-3, other=2e-4, rel999=3e-5, rel_mean=1e-6, inv_frac=1e-3, inv_med=4e-7,
                      res_rel999=3e-5, res_rel_mean=1e-6),
    # [0, 2.6e-3, 3.3e-5, 0, 0, 0, 1.6e-7, 0, 0]
    "fast": dict(m1_begin=0.4,            # [0.29, heightfield: approximate normalisation moves more cosines]
                 m1_spatial=5e-3,         # [2.7e-3]
                 other=8e-4,              # [2.7e-4 (10 pixels), heightfield, frame_begin]
                 rel999=3e-5,             # [1.2e-5]
                 rel_mean=1e-6,           # [2.3e-7]
                 inv_frac=1e-3,           # [0]
                 inv_med=4e-7,            # [1.7e-7]
                 res_rel999=3e-5,         # [1.2e-5]
                 res_rel_mean=1e-6),      # [2.2e-7]
}


@pytest.fixture(scope="module")
def rt():
    r = cedecrt.Runtime(0)
    yield r
    r.close()


def lit_blocks_ao():
    t = small_scene("blocks_ao").copy()
    t["emissive"][100:140] = (5.0, 4.0, 3.0)
    return t


def bumps():
    """a seeded heightfield: normals that vary from pixel to pixel (the blocks scenes have axis-aligned normals only,
    on which the rejection heuristics' cosine power is 0 or 1 whatever its exponent), 3 % of its triangles emissive"""
    rng = np.random.default_rng(21)
    n = 40
    xs = np.linspace(-8.0, 8.0, n + 1)
    X, Z = np.meshgrid(xs, xs, indexing="ij")
    Y = 0.8 * np.sin(0.9 * X) * np.cos(0.7 * Z) + rng.uniform(-0.15, 0.15, X.shape)
    P = np.stack([X, Y, Z], -1).astype(np.float32)
    a, b, c, d = P[:-1, :-1], P[1:, :-1], P[1:, 1:], P[:-1, 1:]
    v = np.concatenate([np.stack([a, c, b], 2).reshape(-1, 3, 3), np.stack([a, d, c], 2).reshape(-1, 3, 3)])
    tris = np.zeros(len(v), cedecrt.TRIANGLE)
    tris["vertices"] = v
    tris["color"] = rng.uniform(0.3, 0.9, (len(v), 3)).astype(np.float32)
    lit = rng.random(len(v)) < 0.03
    tris["emissive"][lit] = rng.uniform(2.0, 12.0, (int(lit.sum()), 3)).astype(np.float32)
    return tris


# name -> (triangles, camera, W, H, rows the device and the oracle compute: (y0, y1) or None for all)
SCENES = {
    "blocks_ao_lit_320x180": lambda: (lit_blocks_ao(), CAM_AO, 320, 180, None),
    "blocks_restir_band": lambda: (scene("blocks_restir"), CAM_RESTIR, 1920, 1080, (600, 616)),
    "ragged_257x9": lambda: (lit_blocks_ao(), CAM_AO, 257, 9, None),
    "bumps_320x180": lambda: (bumps(), CAM_BUMPS, 320, 180, None),
}


class Tap:
    """the oracle with the input and output of every stage of one frame recorded (orc.RestirChain drives it)"""

    def __init__(self, o):
        self.o, self.log = o, {}

    def __getattr__(self, name):
        return getattr(self.o, name)

    def temporal_resampling(self, W, H, frame, g, tris, vis, eye, opt, prev, res):
        self.log["history"] = prev.copy()
        return self.o.temporal_resampling(W, H, frame, g, tris, vis, eye, opt, prev, res)

    def save_temporal_reservoir(self, W, H, src, dst):
        self.o.save_temporal_reservoir(W, H, src, dst)
        self.log["begin"] = dst.copy()
        return dst

    def spatial_resampling(self, W, H, frame, pas, g, tris, vis, eye, opt, rin, rout):
        self.log["in", pas] = rin.copy()
        self.o.spatial_resampling(W, H, frame, pas, g, tris, vis, eye, opt, rin, rout)
        self.log["out", pas] = rout.copy()
        return rout

    def resolve(self, accum, W, H, g, tris, vis, eye, opt, res):
        self.log["accum_in"] = accum.copy()
        self.o.resolve(accum, W, H, g, tris, vis, eye, opt, res)
        self.log["accum"] = accum.copy()
        return accum


def oracle_frame(port, tris, cam, W, H, rows, kw, warm=2):
    """the oracle's stage inputs and outputs of frame warm + 1 (exact arithmetic)"""
    tap = Tap(port)
    port.set_math_mode(1)
    if rows:
        port.set_range(rows[0] * W, rows[1] * W)
    g = port.geom_build(tris)
    try:
        ch = orc.RestirChain(tap, W, H, tris, g, *cam, orc.make_options(**kw))
        for _ in range(warm + 1):
            tap.log = {}
            ch.step()
        tap.log["vis"] = ch.vis.copy()
        tap.log["frame"] = ch.frame
        return tap.log
    finally:
        port.geom_free(g)
        port.set_range(0, -1)


def skip_mask(vis, tris):
    idx = vis["index"]
    em = (tris["emissive"] > 0).any(1)
    s = idx < 0
    s[~s] = em[idx[~s]]
    return s


def pixel_surface(vis, tris, eye):
    """surface_from_visibility (restir_core.cuh) in float64: point, normal turned towards the eye"""
    v = tris["vertices"][np.maximum(vis["index"], 0)].astype(np.float64)
    u, w = vis["uv"][:, 0].astype(np.float64)[:, None], vis["uv"][:, 1].astype(np.float64)[:, None]
    p = (1.0 - u - w) * v[:, 0] + u * v[:, 1] + w * v[:, 2]
    n = np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0])
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    n[((np.asarray(eye, np.float64) - p) * n).sum(1) < 0] *= -1.0
    return p, n


def invariant_deviation(res, p, n):
    """|ucw * M * p_hat / w_sum - 1| with p_hat the target function (reservoir.hpp:42-59, restir_core.cuh) of the stored
    sample at the pixel's surface, in float64; NaN where the target or w_sum is zero (nothing to check)"""
    hp, hn, rad = (res[f].astype(np.float64) for f in ("hit_position", "hit_normal", "radiance"))
    d = hp - p
    sqr = (d * d).sum(1)
    with np.errstate(divide="ignore", invalid="ignore"):
        dn = d / np.sqrt(sqr)[:, None]
        g = np.abs((dn * n).sum(1)) * np.abs((-dn * hn).sum(1)) / sqr
        p_hat = (1.0 / np.float64(np.float32(np.pi))) * g * (rad @ np.array([0.1762044, 0.8129847, 0.0108109]))
        w_sum = res["w_sum"].astype(np.float64)
        dev = np.abs(res["ucw"].astype(np.float64) * res["M"] * p_hat / w_sum - 1.0)
    dev[~((p_hat > 0) & (w_sum > 0) & np.isfinite(p_hat))] = np.nan
    return dev


def rel_err(a, b):
    a, b = a.astype(np.float64).reshape(len(a), -1), b.astype(np.float64).reshape(len(b), -1)
    return (np.abs(a - b) / np.maximum(np.abs(b), 1e-30)).max(1)


def compare_reservoirs(dev, ref):
    """per-stage statistics of diffuse pixels: decision flips, and the relative error of the pixels that decided alike"""
    hp_d, hp_r = dev["hit_position"].astype(np.float64), ref["hit_position"].astype(np.float64)
    close = np.abs(hp_d - hp_r).max(1) <= 1e-4 * np.maximum(np.abs(hp_r).max(1), 1.0)
    alike = (dev["M"] == ref["M"]) & (dev["visibility"] == ref["visibility"]) & close
    e = np.concatenate([rel_err(dev[f][alike], ref[f][alike]) for f in ("w_sum", "ucw", "radiance")])
    # M alone one apart: the same sample and visibility, the merge's truncation trunc(M * w) landed on the other integer
    m1 = (np.abs(dev["M"].astype(np.int64) - ref["M"]) == 1) & (dev["visibility"] == ref["visibility"]) & close
    flip = float(1.0 - alike.mean())
    return dict(alike=alike, flip=flip, flip_m1=float(m1.mean()), flip_other=float((~alike & ~m1).mean()),
                rel999=float(np.quantile(e, 0.999)) if len(e) else 0.0, rel_mean=float(e.mean()) if len(e) else 0.0,
                rel_max=float(e.max()) if len(e) else 0.0)


def invariant_stats(res, p, n):
    dev = invariant_deviation(res, p, n)
    dev = dev[np.isfinite(dev)]
    return dict(inv_n=len(dev), inv_frac=float((dev > 1e-3).mean()), inv_med=float(np.median(dev)))


def patch_skip(buf, n, skip):
    """crt_reservoir_import_aos writes plain records; the fused frame marks sky / emissive pixels inside the record
    (restir_fast.cuh: store_skip, plane 0 of the sector-planar layout), and a spatial pass skips such neighbours"""
    raw = buf.to_host().view(np.uint8).copy()
    plane0 = raw[:32 * n].view(np.uint32).reshape(n, 8)
    plane0[skip] = 0
    plane0[skip, 6] = K_SKIP
    buf.upload(raw)


def device_frame(rt, mode, tris, cam, W, H, rows, kw, log):
    """every stage of the fused frame in `mode`, each from the oracle's input of that stage"""
    n = W * H
    eye = tuple(float(np.float32(v)) for v in cam[0])
    raygen = cedecrt.lookat(cam[0], cam[1], W, H)
    d_tris = rt.to_device(tris)
    geom = rt.build_geometry(d_tris)
    lights = rt.to_device(cedecrt.light_indices(tris))
    opt = cedecrt.Options(**kw)
    pix, acc, vis = rt.buffer(np.uint8, 4 * n), rt.buffer(cedecrt.FLOAT4, n), rt.buffer(cedecrt.VISIBILITY, n)
    r0, r1, temporal = (rt.buffer(cedecrt.RESERVOIR, n) for _ in range(3))
    bufs = rt.restir_buffers(pix, acc, vis, r0, r1, temporal)
    tmp = rt.buffer(cedecrt.RESERVOIR, n)
    skip = skip_mask(log["vis"], tris)

    def load(arr, dst, mark_skip):
        rt.reservoir_import_aos(W, H, rt.to_device(arr), dst)
        if mark_skip:
            patch_skip(dst, n, skip)

    def export(src):
        rt.reservoir_export_aos(W, H, src, tmp)
        return tmp.to_host()

    out = {}
    rt.set_math_mode(mode)
    if rows:
        rt.set_row_range(*rows)
    try:
        load(log["history"], temporal, False)
        rt.restir_frame_begin(W, H, log["frame"], geom, d_tris, raygen, eye, lights, opt, bufs)
        out["vis"] = vis.to_host()
        out["begin"] = export(temporal)
        passes = opt.spatial_resampling_passes
        for k in range(passes):
            src, dst = (temporal, r1) if k == 0 else (r1, r0) if k % 2 else (r0, r1)
            load(log["in", k], src, True)
            rt.restir_spatial_pass(W, H, log["frame"], k, geom, d_tris, eye, opt, bufs)
            out["out", k] = export(dst)
        final = r1 if passes % 2 else r0
        load(log["out", passes - 1], final, True)
        acc.upload(log["accum_in"])
        rt.restir_frame_end(W, H, geom, d_tris, eye, opt, bufs)
        out["accum"] = acc.to_host().view(np.float32).reshape(-1, 4)
        out["pixels"] = pix.to_host()
    finally:
        rt.set_row_range(0, -1)
        geom.destroy()
    return out


@pytest.mark.parametrize("name", list(SCENES))
def test_fused_stages_in_every_math_mode_against_the_oracle(rt, port, name):
    """Each stage of the fused frame in EXACT, REFERENCE, LIBDEVICE and FAST mode from the oracle's input state of frame
    3: bit-exact in EXACT; in the others primary visibility, sky and emissive pixels bit-exact, decision flips, the error
    of same-decision pixels and the float64 invariant within the mode's bars (BARS)."""
    tris, cam, W, H, rows = SCENES[name]()
    log = oracle_frame(port, tris, cam, W, H, rows, KW)
    sl = slice((H - rows[1]) * W, (H - rows[0]) * W) if rows else slice(0, W * H)  # bottom-up storage
    vis_ref = log["vis"][sl]
    skip = skip_mask(vis_ref, tris)
    diffuse = ~skip
    assert diffuse.sum() >= 100
    p, nrm = pixel_surface(vis_ref[diffuse], tris, np.float32(cam[0]))
    passes = KW.get("spatial_resampling_passes", 3)
    stages = ["begin"] + [("out", k) for k in range(passes)]
    ref_of = lambda s: log[s][sl]
    report, failures = [], []
    try:
        # the invariant on the oracle's own reservoirs: what the device is held to must hold for the specification too
        for s in stages:
            st = invariant_stats(ref_of(s)[diffuse], p, nrm)
            report.append("%-22s oracle    %-9s invariant: off > 1e-3 %.2e, median %.2e (n %d)" % (
                name, s, st["inv_frac"], st["inv_med"], st["inv_n"]))
            if st["inv_frac"] > BARS["reference"]["inv_frac"] or st["inv_med"] > BARS["reference"]["inv_med"]:
                failures.append(("oracle", s, "invariant", st))
        for mode_name, mode in MODES.items():
            out = device_frame(rt, mode, tris, cam, W, H, rows, KW, log)
            vis = out["vis"][sl]
            assert same(vis["index"], vis_ref["index"]) and same(vis["uv"], vis_ref["uv"]), mode_name
            for s in stages:
                dev, ref = out[s][sl], ref_of(s)
                if s == "begin":  # sky / emissive pixels: Reservoir{}, as save_temporal copies it
                    assert reservoir_mismatch(dev[skip], ref[skip]) == 0, (mode_name, s)
                else:  # the reference leaves them untouched; the fused frame marks them and exports Reservoir{}
                    assert not dev[skip].view(np.uint8).any(), (mode_name, s)
                if mode_name == "exact":
                    assert reservoir_mismatch(dev[diffuse], ref[diffuse]) == 0, (mode_name, s)
                    continue
                st = compare_reservoirs(dev[diffuse], ref[diffuse])
                st.update(invariant_stats(dev[diffuse], p, nrm))
                report.append("%-22s %-9s %-9s flipped: M alone by one %.2e, other %.2e; same-decision rel. error p99.9 %.2e "
                              "mean %.2e max %.2e; invariant: off > 1e-3 %.2e median %.2e" % (
                                  name, mode_name, s, st["flip_m1"], st["flip_other"], st["rel999"], st["rel_mean"],
                                  st["rel_max"], st["inv_frac"], st["inv_med"]))
                # one flipped pixel of slack for small images (the ragged size has 113 diffuse pixels)
                slack = 1.0 / diffuse.sum()
                bars = dict(BARS[mode_name])
                bars["flip_m1"] = bars["m1_begin" if s == "begin" else "m1_spatial"] + slack
                bars["flip_other"] = bars["other"] + slack
                bad = [k for k in ("flip_m1", "flip_other", "rel999", "rel_mean", "inv_frac", "inv_med") if st[k] > bars[k]]
                if bad:
                    failures.append((mode_name, s, bad, {k: v for k, v in st.items() if k != "alike"}))
            acc, acc_ref, acc_in = out["accum"][sl], log["accum"][sl], log["accum_in"][sl]
            assert same(acc[skip], acc_ref[skip]) and same(acc[:, 3], acc_ref[:, 3]), mode_name
            rgba, rgba_ref = out["pixels"].reshape(-1, 4)[sl], port.tone_mapping(out["accum"], W, H).reshape(-1, 4)[sl]
            if mode_name == "exact":
                assert same(acc, acc_ref) and same(rgba, rgba_ref)
                continue
            # tone mapping in the mode's own functions: within one step of the correctly rounded one
            assert np.abs(rgba.astype(np.int32) - rgba_ref).max() <= 1, mode_name
            # resolve: pixels whose final reservoirs decided alike shade alike, unless their shadow ray (its origin rounded
            # in the mode's arithmetic) grazes an edge differently
            alike = compare_reservoirs(out["out", passes - 1][sl][diffuse], ref_of(("out", passes - 1))[diffuse])["alike"]
            e = rel_err((acc - acc_in)[diffuse][alike, :3], (acc_ref - acc_in)[diffuse][alike, :3])
            frac = float((e > 1e-3).mean())
            rest = e[e <= 1e-3]  # the shading of the others: a bias of resolve's own arithmetic shows here
            res999, res_mean = float(np.quantile(rest, 0.999)), float(rest.mean())
            report.append("%-22s %-9s resolve   same-decision pixels off by > 1e-3: %.2e; the others: rel. error p99.9 %.2e "
                          "mean %.2e" % (name, mode_name, frac, res999, res_mean))
            bad = [k for k, v, bar in (("off", frac, BARS[mode_name]["m1_spatial"]), ("rel999", res999, BARS[mode_name]["res_rel999"]),
                                       ("rel_mean", res_mean, BARS[mode_name]["res_rel_mean"])) if v > bar]
            if bad:
                failures.append((mode_name, "resolve", bad, frac, res999, res_mean))
    finally:
        print("\n" + "\n".join(report))
        port.set_math_mode(0)
    assert not failures, failures


# ------------------------------------------------------------------ the own-triangle pre-test under flush-to-zero
def denormal_edge_scene():
    """A floor strip of unit right triangles (y = 0, z in [0, 1], x in [-2, 2]) that ends at the line z = 0, and one
    emissive wall below it in the plane z = -2^-118.  Every coordinate is 0 or a power of two, so light sample points and
    surface points are exact products whatever the arithmetic, and the camera sits in the plane z = 0: the primary rays
    of column W / 2 hit the floor exactly on its edge.  Their visibility rays leave that edge downwards and cross the
    floor's plane at z = -2^-118 * t with t ~ 1e-3: at a denormal distance outside the triangle they start on, which
    the walk (never flushed) rejects.  A pre-test that flushed the sub-area -1e-39 to zero would accept it."""
    tris = []
    for k in (-2, -1, 0, 1):
        tris.append([[k, 0, 0], [k + 1, 0, 0], [k, 0, 1]])          # the edge v0 -> v1 lies on z = 0
        tris.append([[k + 1, 0, 0], [k + 1, 0, 1], [k, 0, 1]])
    c = 2.0 ** -118
    wall = [[[-2, -2, -c], [2, -2, -c], [2, -0.5, -c]], [[-2, -2, -c], [2, -0.5, -c], [-2, -0.5, -c]]]
    out = np.zeros(len(tris) + 2, cedecrt.TRIANGLE)
    out["vertices"] = np.array(tris + wall, np.float32)
    out["color"] = 0.5
    out["emissive"][-2:] = (8.0, 8.0, 8.0)
    return out


def own_triangle_scene():
    """test_gpu_edges.py's case: blocks_ao lit by one triangle below most surfaces, so that most visibility rays start
    on the triangle that stops them or leave it at a grazing angle"""
    tris = small_scene("blocks_ao").copy()
    tris["emissive"][:] = 0
    tris["emissive"][int(np.argmin(tris["vertices"][:, :, 1].mean(axis=1)))] = (30.0, 30.0, 30.0)
    return tris


@pytest.mark.parametrize("mode", ["reference", "fast"])
@pytest.mark.parametrize("name", ["denormal_edge", "own_triangle"])
def test_visibility_of_identical_shadow_rays_equals_the_oracle(rt, port, name, mode):
    """segment_hits_triangle (bvh.cuh) decides some visibility-reuse rays inside the candidate kernel, which the
    REFERENCE and FAST modes compile with contraction and (FAST) flush-to-zero.  Wherever the device's ray is the
    oracle's bit for bit — same surface point and normal, same light sample point, and an offset origin p + 1e-3 n that
    rounds alike with and without contraction — its visibility must be the oracle's."""
    if name == "denormal_edge":
        tris, cam, W, H = denormal_edge_scene(), ((3.0, 2.0, 0.0), (-1.0, 0.0, 0.0)), 64, 48
    else:
        tris, cam, W, H = own_triangle_scene(), CAM_AO, 96, 54
    kw = dict(KW, use_spatial_resampling=0)
    port.set_math_mode(1)
    g = port.geom_build(tris)
    try:
        ch = orc.RestirChain(port, W, H, tris, g, *cam, orc.make_options(**kw))
        ch.step()
        rt.set_math_mode(MODES[mode])
        app = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(**kw), fused=True)
        app.frame()
        dev, ref = app.export_aos(app.temporal), ch.temporal
    finally:
        port.geom_free(g)
        port.set_math_mode(0)
    diffuse = ~skip_mask(ch.vis, tris)
    bits = lambda r, f: r[f].view(np.uint32)
    ident = diffuse & (dev["M"] == ref["M"])
    for f in ("origin_position", "origin_normal", "hit_position"):
        ident &= (bits(dev, f) == bits(ref, f)).all(1)
    p, nrm = ref["origin_position"], ref["origin_normal"]
    off = np.float32(0.001) * nrm
    org_sep = (p + off).astype(np.float32)
    org_fma = (p.astype(np.float64) + np.float64(np.float32(0.001)) * nrm.astype(np.float64)).astype(np.float32)
    ident &= (org_sep.view(np.uint32) == org_fma.view(np.uint32)).all(1)
    wrong = ident & (dev["visibility"] != ref["visibility"])
    print("%s, %s: %d diffuse pixels, %d with the oracle's shadow ray bit for bit, %d of them visible, %d flags differ" % (
        name, mode, int(diffuse.sum()), int(ident.sum()), int((ident & (ref["visibility"] == 1)).sum()), int(wrong.sum())))
    assert ident.sum() >= 20
    if name == "denormal_edge":
        # the rays that leave the floor's edge (column W / 2) are the ones the scene is for: visible in the oracle
        edge = np.zeros((H, W), bool)
        edge[:, W // 2] = True
        edge = edge.reshape(-1) & ident & (ref["origin_position"][:, 2] == 0) & (ref["visibility"] == 1)
        assert edge.sum() >= 5, int(edge.sum())
    assert wrong.sum() == 0, np.nonzero(wrong)[0][:20]
