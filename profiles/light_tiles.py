"""Cost and noise of presampled light tiles (crt_set_light_tiles) for the ReSTIR DI candidates.

One GPU command:
  * frame time (CUDA events) and per-kernel times (crt_profile_begin/end) of the fused 10_restir_di frame at 3840x2160 on
    BASELINE config 5 (the procedural stand-in when the blocks_restir cache is absent; the output names the scene), arms
    alternated over several rounds: uniform, power with K = 2^22, power + tiles and uniform + tiles at several (T, S);
  * the tile build's time (the light_tiles kernel, once per frame);
  * noise at 1920x1080: relative MSE of the F-frame accumulation (F = 1, 16, 64) against a long accumulation of the same
    arm, at equal frames and — using the measured frame times and MSE ~ 1/F — at equal GPU time;
  * the device's name and power limit (read-only nvidia-smi query) beside the numbers.
Writes JSON (default profiles/light_tiles/light_tiles.json)."""
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

U, P = cedecrt.LIGHTS_UNIFORM, cedecrt.LIGHTS_POWER
# (name, light mode, log2 K, (log2 T, log2 S))
ARMS = (("uniform", U, 0, (0, 0)), ("power_2^22", P, 22, (0, 0)), ("power_2^22+tiles_7_10", P, 22, (7, 10)),
        ("uniform+tiles_7_10", U, 0, (7, 10)), ("power_2^22+tiles_5_10", P, 22, (5, 10)),
        ("power_2^22+tiles_9_10", P, 22, (9, 10)), ("power_2^22+tiles_7_8", P, 22, (7, 8)))


def set_arm(rt, arm):
    _, mode, log2, tiles = arm
    rt.set_light_sampling(mode, log2)
    rt.set_light_tiles(*tiles)


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
        for arm in arms:
            set_arm(rt, arm)
            for _ in range(warmup):
                app.frame()
            rt.timer_start()
            for _ in range(frames):
                app.frame()
            out[arm[0]].append(rt.timer_stop_ms() / frames)
    return out


def kernel_times(rt, app, arms, frames=5):
    res = {}
    for arm in arms:
        set_arm(rt, arm)
        app.frame()
        rt.profile_begin()
        for _ in range(frames):
            app.frame()
        prof = rt.profile_end()
        agg = {}
        for k, ms in prof:
            agg[k] = agg.get(k, 0.0) + ms / frames
        res[arm[0]] = {k: round(v, 4) for k, v in agg.items()}
    return res


def rel_mse(img, ref):
    return float(((img - ref) ** 2).mean() / (ref ** 2).mean())


def accum_image(buf):
    a = buf.to_host().view(np.float32).reshape(-1, 4)
    return a[:, :3] / a[:, 3:4]


def noise_restir(rt, tris, cam, W, H, arms, checkpoints, ref_frames):
    out = {}
    for arm in arms:
        set_arm(rt, arm)
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
        out[arm[0]] = {"ms_per_frame": ms / ref_frames, "ref_frames": ref_frames, "ref": ref,
                       "rel_mse": {f: rel_mse(snaps[f], ref) for f in checkpoints}}
        app.geom.destroy()
        print("restir", arm[0], "%.1f s" % (time.time() - t0), flush=True)
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "light_tiles", "light_tiles.json"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--ref-frames", type=int, default=1024)
    args = ap.parse_args()
    import bench

    tris, cam, workload = bench.load_workload()
    lights = cedecrt.light_indices(tris)
    rt = cedecrt.Runtime(0)  # CRT_MATH_REFERENCE, the default
    result = {"device": rt.device_name(), "nvidia_smi": gpu_info(), "workload": workload, "triangles": int(len(tris)),
              "lights": int(len(lights)), "math_mode": "REFERENCE", "arms": {a[0]: {"lights": "power" if a[1] else "uniform",
              "log2_slots": a[2], "log2_tiles": a[3][0], "log2_tile_size": a[3][1]} for a in ARMS}}
    print(result, flush=True)
    W, H = 3840, 2160
    app = cedecrt.RestirDI(rt, W, H, tris, *cam, cedecrt.Options(accumulate=1, use_temporal_resampling=1,
                                                                 use_spatial_resampling=1), fused=True)
    for arm in ARMS:  # build every arm's tables once before timing
        set_arm(rt, arm)
        app.frame()
    rt.sync()
    ft = frame_times(rt, app, ARMS, args.rounds, args.frames, 3)
    result["frame_ms_4k"] = {k: {"median": float(np.median(v)), "all": v} for k, v in ft.items()}
    print("frame ms", result["frame_ms_4k"], flush=True)
    result["kernel_ms_4k"] = kernel_times(rt, app, ARMS)
    print("kernel ms", result["kernel_ms_4k"], flush=True)
    app.geom.destroy()
    del app
    cps = (1, 16, 64)
    W, H = 1920, 1080
    result["noise_1080p"] = {"10_restir_di": summarise(noise_restir(rt, tris, cam, W, H, ARMS, cps, args.ref_frames), cps)}
    result["noise_reference"] = {"10_restir_di": "%d-frame accumulation of the same arm" % args.ref_frames}
    rt.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1, default=float)
    print(json.dumps(result, default=float)[:6000])


if __name__ == "__main__":
    main()
