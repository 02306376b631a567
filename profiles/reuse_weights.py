"""Cost and effect of the unbiased reuse weights (crt_set_reuse_weights) against the reference's.

One GPU command:
  * frame time (CUDA events) of the fused 10_restir_di frame at 3840x2160 on bench.py's workload (the procedural
    stand-in when the blocks_restir cache is absent; the output names the scene), CRT_MATH_REFERENCE, the two modes
    alternated over several rounds; per-kernel times (crt_profile_begin/end) of candidate_temporal and spatial_fast;
  * DESIGN.md section 14's open question: 2048-frame 1920x1080 references with temporal and spatial reuse, uniform
    against power light selection, in each weight mode: the relative MSE between the two references;
  * noise: relative MSE of the F-frame accumulation (F = 1, 16, 64) against the long reference of the same arm;
  * the device's name and power limit (read-only nvidia-smi query) beside the numbers.
Writes JSON (default profiles/reuse_weights/reuse_weights.json)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "cedec-2024-rt_b200", "python"))

import cedecrt  # noqa: E402

MODES = (("reference", cedecrt.REUSE_REFERENCE), ("unbiased", cedecrt.REUSE_UNBIASED))
LIGHTS = (("uniform", cedecrt.LIGHTS_UNIFORM), ("power", cedecrt.LIGHTS_POWER))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def frame_times(rt, app, rounds, frames, warmup):
    out = {m[0]: [] for m in MODES}
    for _ in range(rounds):
        for name, mode in MODES:
            rt.set_reuse_weights(mode)
            for _ in range(warmup):
                app.frame()
            rt.timer_start()
            for _ in range(frames):
                app.frame()
            out[name].append(rt.timer_stop_ms() / frames)
    return out


def kernel_times(rt, app, frames=5):
    res = {}
    for name, mode in MODES:
        rt.set_reuse_weights(mode)
        app.frame()
        rt.profile_begin()
        for _ in range(frames):
            app.frame()
        agg = {}
        for k, ms in rt.profile_end():
            agg[k] = agg.get(k, 0.0) + ms / frames
        res[name] = {k: round(v, 4) for k, v in agg.items()}
    return res


def rel_mse(img, ref):
    return float(((img - ref) ** 2).mean() / (ref ** 2).mean())


def accum_image(buf):
    a = buf.to_host().view(np.float32).reshape(-1, 4)
    return a[:, :3] / a[:, 3:4]


def references(rt, tris, cam, W, H, checkpoints, ref_frames):
    out, refs = {}, {}
    for lname, lmode in LIGHTS:
        for mname, mmode in MODES:
            rt.set_light_sampling(lmode)
            rt.set_reuse_weights(mmode)
            app = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(accumulate=1, use_temporal_resampling=1,
                                                                         use_spatial_resampling=1), fused=True)
            snaps, t0 = {}, time.time()
            rt.timer_start()
            for f in range(1, ref_frames + 1):
                app.frame()
                if f in checkpoints:
                    snaps[f] = accum_image(app.accumulation)
            ms = rt.timer_stop_ms()
            refs[lname, mname] = accum_image(app.accumulation)
            out["%s/%s" % (lname, mname)] = {"ms_per_frame": ms / ref_frames,
                                             "rel_mse_vs_own_reference": {f: rel_mse(snaps[f], refs[lname, mname])
                                                                          for f in checkpoints}}
            app.geom.destroy()
            print(lname, mname, "%.1f s" % (time.time() - t0), flush=True)
    rt.set_light_sampling(cedecrt.LIGHTS_UNIFORM)
    rt.set_reuse_weights(cedecrt.REUSE_REFERENCE)
    gap = {m: rel_mse(refs["power", m], refs["uniform", m]) for m, _ in MODES}
    # how far each weight mode's reference lies from the other's, per light selection
    cross = {l: rel_mse(refs[l, "unbiased"], refs[l, "reference"]) for l, _ in LIGHTS}
    mean = {"%s/%s" % k: float(v.mean()) for k, v in refs.items()}
    return out, gap, cross, mean


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "reuse_weights", "reuse_weights.json"))
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--ref-frames", type=int, default=2048)
    args = ap.parse_args()
    import bench

    tris, cam, workload = bench.load_workload()
    rt = cedecrt.Runtime(0)  # CRT_MATH_REFERENCE, the default
    result = {"device": rt.device_name(), "nvidia_smi": gpu_info(), "workload": workload, "triangles": int(len(tris)),
              "math_mode": "REFERENCE"}
    print(result, flush=True)
    W, H = 3840, 2160
    app = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(accumulate=1, use_temporal_resampling=1,
                                                                 use_spatial_resampling=1), fused=True)
    for _, mode in MODES:
        rt.set_reuse_weights(mode)
        app.frame()
    rt.sync()
    ft = frame_times(rt, app, args.rounds, args.frames, 3)
    result["frame_ms_4k"] = {k: {"median": float(np.median(v)), "all": v} for k, v in ft.items()}
    print("frame ms", result["frame_ms_4k"], flush=True)
    km = kernel_times(rt, app)
    result["kernel_ms_4k"] = km
    result["kernel_ms_4k_summary"] = {k: {m: km[m].get(k) for m, _ in MODES} for k in ("candidate_temporal", "spatial_fast")}
    print("kernel ms", result["kernel_ms_4k_summary"], flush=True)
    app.geom.destroy()
    del app
    cps = (1, 16, 64)
    out, gap, cross, mean = references(rt, tris, cam, 1920, 1080, cps, args.ref_frames)
    result["noise_1080p"] = out
    result["uniform_vs_power_reference_rel_mse"] = gap
    result["unbiased_vs_reference_weights_rel_mse"] = cross
    result["reference_image_mean"] = mean
    result["reference_frames"] = args.ref_frames
    rt.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1, default=float)
    print(json.dumps(result, default=float)[:4000])


if __name__ == "__main__":
    main()
