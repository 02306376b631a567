"""Cost of unbiased reuse weights with a moving camera (crt_restir_set_previous_frame) against the two paths a host with a
moving camera had before: the reference's weights with reprojection, and unbiased weights without reprojection.

One GPU command: the fused 10_restir_di frame at 3840x2160 on bench.py's workload (the procedural stand-in when the
blocks_restir cache is absent; the output names the scene), CRT_MATH_REFERENCE, the camera panning a fixed step per
frame (the accumulation cleared on every move, like the reference's loop).  Three arms, alternated over several rounds:
  reference_reproject   CRT_REUSE_REFERENCE, RestirDI(reproject=True)      (crt_restir_set_previous_camera)
  unbiased              CRT_REUSE_UNBIASED, no reprojection                 (the history read at the same pixel)
  unbiased_reproject    CRT_REUSE_UNBIASED, RestirDI(reproject="surfaces") (crt_restir_set_previous_frame)
Reports the median frame time (CUDA events) and the per-kernel times of crt_profile (candidate_temporal among them), with
the device's name and power limit (read-only nvidia-smi query) read in the same run.
Writes JSON (default profiles/reuse_reprojection/reuse_reprojection.json)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "cedec-2024-rt_b200", "python"))

import cedecrt  # noqa: E402

ARMS = (("reference_reproject", cedecrt.REUSE_REFERENCE, True), ("unbiased", cedecrt.REUSE_UNBIASED, False),
        ("unbiased_reproject", cedecrt.REUSE_UNBIASED, "surfaces"))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


class Pan:
    """one arm's application; every frame moves eye and look-at point by `step`"""

    def __init__(self, rt, tris, cam, W, H, reuse, reproject, step):
        self.rt, self.reuse = rt, reuse
        self.eye, self.center, self.step = np.array(cam[0]), np.array(cam[1]), np.array(step)
        opt = cedecrt.Options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
        self.app = cedecrt.RestirDI(rt, W, H, tris, *cam, opt, fused=True, reproject=reproject)

    def frame(self):
        self.rt.set_reuse_weights(self.reuse)
        self.eye, self.center = self.eye + self.step, self.center + self.step
        self.app.set_camera(tuple(self.eye), tuple(self.center))
        self.app.frame()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "reuse_reprojection", "reuse_reprojection.json"))
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--step", type=float, nargs=3, default=(0.05, 0.0, -0.05))
    args = ap.parse_args()
    import bench

    tris, cam, workload = bench.load_workload()
    rt = cedecrt.Runtime(0)  # CRT_MATH_REFERENCE, the default
    result = {"device": rt.device_name(), "nvidia_smi": gpu_info(), "workload": workload, "triangles": int(len(tris)),
              "math_mode": "REFERENCE", "camera_step_per_frame": list(args.step)}
    print(result, flush=True)
    W, H = 3840, 2160
    arms = {name: Pan(rt, tris, cam, W, H, reuse, rep, args.step) for name, reuse, rep in ARMS}
    for a in arms.values():
        for _ in range(3):
            a.frame()
    rt.sync()
    times = {name: [] for name in arms}
    for _ in range(args.rounds):
        for name, a in arms.items():
            for _ in range(3):
                a.frame()
            rt.timer_start()
            for _ in range(args.frames):
                a.frame()
            times[name].append(rt.timer_stop_ms() / args.frames)
    result["frame_ms_4k"] = {k: {"median": float(np.median(v)), "all": v} for k, v in times.items()}
    print("frame ms", {k: v["median"] for k, v in result["frame_ms_4k"].items()}, flush=True)
    km = {}
    for name, a in arms.items():
        a.frame()
        rt.profile_begin()
        for _ in range(5):
            a.frame()
        agg = {}
        for k, ms in rt.profile_end():
            agg[k] = agg.get(k, 0.0) + ms / 5
        km[name] = {k: round(v, 4) for k, v in agg.items()}
    result["kernel_ms_4k"] = km
    result["candidate_temporal_ms_4k"] = {name: km[name].get("candidate_temporal") for name in arms}
    print("candidate_temporal ms", result["candidate_temporal_ms_4k"], flush=True)
    for a in arms.values():
        a.app.geom.destroy()
    rt.set_reuse_weights(cedecrt.REUSE_REFERENCE)
    rt.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1, default=float)
    print(json.dumps(result, default=float)[:3000])


if __name__ == "__main__":
    main()
