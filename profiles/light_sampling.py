"""Cost and noise of power-proportional light selection (crt_set_light_sampling) against uniform selection.

One GPU command:
  * frame time (CUDA events) and per-kernel times (crt_profile_begin/end) of the fused 10_restir_di frame at 3840x2160 on
    BASELINE config 5 (the procedural stand-in when the blocks_restir cache is absent; the output names the scene), three
    arms alternated over several rounds: uniform, power with the default K, power with K = 2^20;
  * the slot table's build time at that scene's light count;
  * noise at 1920x1080: relative MSE of the F-frame accumulation (F = 1, 4, 16, 64) against a long accumulation of the
    same mode, for 10_restir_di with default options and for 08_nee and 09_ris, per arm, at equal frames and — using the
    measured frame times and MSE ~ 1/F — at equal GPU time;
  * the device's name and power limit (read-only nvidia-smi query) beside the numbers.
Writes JSON (default profiles/light_sampling/light_sampling.json)."""
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

ARMS = (("uniform", cedecrt.LIGHTS_UNIFORM, 0), ("power_default", cedecrt.LIGHTS_POWER, 0), ("power_2^20", cedecrt.LIGHTS_POWER, 20))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def frame_times(rt, app, arms, rounds, frames, warmup):
    out = {a[0]: [] for a in arms}
    for _ in range(rounds):
        for name, mode, log2 in arms:
            rt.set_light_sampling(mode, log2)
            for _ in range(warmup):
                app.frame()
            rt.timer_start()
            for _ in range(frames):
                app.frame()
            out[name].append(rt.timer_stop_ms() / frames)
    return out


def kernel_times(rt, app, arms, frames=5):
    res = {}
    for name, mode, log2 in arms:
        rt.set_light_sampling(mode, log2)
        app.frame()
        rt.profile_begin()
        for _ in range(frames):
            app.frame()
        prof = rt.profile_end()
        agg = {}
        for k, ms in prof:
            agg[k] = agg.get(k, 0.0) + ms / frames
        res[name] = {k: round(v, 4) for k, v in agg.items()}
        # the table build alone (the allocation is kept): drop the cached table and time the next frame's build kernels
        builds = []
        for _ in range(3):
            rt.lights_changed(app.geom)
            rt.profile_begin()
            app.frame()
            prof = rt.profile_end()
            builds.append(sum(ms for k, ms in prof if k.startswith("light_") or k == "build_light_table"))
        res[name]["table_build_ms"] = round(float(np.median(builds)), 4)
    return res


def rel_mse(img, ref):
    return float(((img - ref) ** 2).mean() / (ref ** 2).mean())


def accum_image(buf):
    a = buf.to_host().view(np.float32).reshape(-1, 4)
    return a[:, :3] / a[:, 3:4]


def noise_restir(rt, tris, cam, W, H, arms, checkpoints, ref_frames):
    out = {}
    for name, mode, log2 in arms:
        rt.set_light_sampling(mode, log2)
        app = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(accumulate=1, use_temporal_resampling=1,
                                                                     use_spatial_resampling=1), fused=True)
        snaps, t0 = {}, time.time()
        rt.timer_start()
        for f in range(1, ref_frames + 1):
            app.frame()
            if f in checkpoints:
                snaps[f] = accum_image(app.accumulation)
        ms = rt.timer_stop_ms()
        ref = accum_image(app.accumulation)
        out[name] = {"ms_per_frame": ms / ref_frames, "ref_frames": ref_frames, "ref": ref,
                     "rel_mse": {f: rel_mse(snaps[f], ref) for f in checkpoints}}
        app.geom.destroy()
        print("restir", name, "%.1f s" % (time.time() - t0), flush=True)
    return out


def noise_paths(rt, example, tris, cam, W, H, arms, checkpoints, ref_frames, options):
    out = {}
    d_t, d_l = rt.to_device(tris), rt.to_device(cedecrt.light_indices(tris))
    g = rt.build_geometry(d_t)
    rg = cedecrt.lookat(*cam, W, H)
    acc = rt.buffer(cedecrt.FLOAT4, W * H)
    for name, mode, log2 in arms:
        rt.set_light_sampling(mode, log2)
        rt.clear(acc, W, H)
        snaps = {}
        rt.timer_start()
        for f in range(1, ref_frames + 1):
            rt.path_trace(example, W, H, f, g, d_t, d_l, rg, options, acc)
            if f in checkpoints:
                snaps[f] = accum_image(acc)
        ms = rt.timer_stop_ms()
        ref = accum_image(acc)
        out[name] = {"ms_per_frame": ms / ref_frames, "ref_frames": ref_frames, "ref": ref,
                     "rel_mse": {f: rel_mse(snaps[f], ref) for f in checkpoints}}
    g.destroy()
    return out


def summarise(noise, checkpoints):
    """equal frames: MSE ratio power / uniform; equal GPU time: the same ratio times the frame-time ratio (MSE ~ 1/F)"""
    u = noise["uniform"]
    for name, arm in noise.items():
        arm["ref_rel_diff_vs_uniform_ref"] = rel_mse(arm["ref"], u["ref"])
        t = arm["ms_per_frame"] / u["ms_per_frame"]
        arm["mse_ratio_equal_frames"] = {f: arm["rel_mse"][f] / u["rel_mse"][f] for f in checkpoints}
        arm["mse_ratio_equal_time"] = {f: arm["rel_mse"][f] / u["rel_mse"][f] * t for f in checkpoints}
    for arm in noise.values():
        del arm["ref"]
    return noise


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "light_sampling", "light_sampling.json"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--ref-frames", type=int, default=2048)
    ap.add_argument("--path-ref-frames", type=int, default=512)
    args = ap.parse_args()
    import bench

    tris, cam, workload = bench.load_workload()
    lights = cedecrt.light_indices(tris)
    rt = cedecrt.Runtime(0)  # CRT_MATH_REFERENCE, the default
    result = {"device": rt.device_name(), "nvidia_smi": gpu_info(), "workload": workload, "triangles": int(len(tris)),
              "lights": int(len(lights)), "math_mode": "REFERENCE"}
    print(result, flush=True)
    W, H = 3840, 2160
    app = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(accumulate=1, use_temporal_resampling=1,
                                                                 use_spatial_resampling=1), fused=True)
    for name, mode, log2 in ARMS:  # build every arm's table once before timing
        rt.set_light_sampling(mode, log2)
        app.frame()
    rt.sync()
    ft = frame_times(rt, app, ARMS, args.rounds, args.frames, 3)
    result["frame_ms_4k"] = {k: {"median": float(np.median(v)), "all": v} for k, v in ft.items()}
    print("frame ms", result["frame_ms_4k"], flush=True)
    result["kernel_ms_4k"] = kernel_times(rt, app, ARMS)
    print("kernel ms", result["kernel_ms_4k"], flush=True)
    app.geom.destroy()
    del app
    cps = (1, 4, 16, 64)
    W, H = 1920, 1080
    noise = {"10_restir_di": summarise(noise_restir(rt, tris, cam, W, H, ARMS, cps, args.ref_frames), cps)}
    print("restir noise done", flush=True)
    for ex, opt in ((8, cedecrt.Options(accumulate=1, max_depth=4)),
                    (9, cedecrt.Options(accumulate=1, max_depth=4, ris_sample_count=32))):
        noise["%02d" % ex] = summarise(noise_paths(rt, ex, tris, cam, W, H, ARMS, cps, args.path_ref_frames, opt), cps)
        print(ex, "noise done", flush=True)
    result["noise_1080p"] = noise
    result["noise_reference"] = {"10_restir_di": "%d-frame accumulation of the same arm" % args.ref_frames,
                                 "08/09": "%d-frame accumulation of the same arm" % args.path_ref_frames}
    rt.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1, default=float)
    print(json.dumps(result, default=float)[:4000])


if __name__ == "__main__":
    main()
