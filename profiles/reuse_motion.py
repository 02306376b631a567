"""Cost of reprojection that follows moving geometry (RestirDI.set_triangles: crt_restir_set_previous_triangles) against
the static assumption a host that refits every frame had before.

One GPU command: the fused 10_restir_di frame at 3840x2160 on bench.py's workload (the procedural stand-in when the
blocks_restir cache is absent; the output names the scene), CRT_MATH_REFERENCE, a share of the non-emissive triangles
(runs of 12, every 8th run) moving up and back down by a fixed step on alternate frames, crt_refit_geometry every frame.
Three arms, alternated over several rounds:
  static               CRT_REUSE_UNBIASED, RestirDI(reproject="surfaces"), the vertices uploaded and the tree refitted
                       behind RestirDI's back (the previous frame's look-up on this frame's triangles)
  motion_reference     CRT_REUSE_REFERENCE, RestirDI(reproject=True).set_triangles
  motion_unbiased      CRT_REUSE_UNBIASED, RestirDI(reproject="surfaces").set_triangles
Each frame is timed on its own with CUDA events, the vertex upload and the refit outside the window; reports the median
frame time, the per-kernel times of crt_profile (candidate_temporal among them) and the refit time of crt_geometry_stats,
with the device's name and power limit (read-only nvidia-smi query) read in the same run.
Writes JSON (default profiles/reuse_motion/reuse_motion.json)."""
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

ARMS = (("static", cedecrt.REUSE_UNBIASED, "surfaces", False), ("motion_reference", cedecrt.REUSE_REFERENCE, True, True),
        ("motion_unbiased", cedecrt.REUSE_UNBIASED, "surfaces", True))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


class Animated:
    """one arm's application; frame() alternates the two vertex states, then renders one timed frame"""

    def __init__(self, rt, states, cam, W, H, reuse, reproject, motion):
        self.rt, self.reuse, self.states, self.motion, self.k = rt, reuse, states, motion, 0
        opt = cedecrt.Options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
        self.app = cedecrt.RestirDI(rt, W, H, states[0], *cam, opt, fused=True, reproject=reproject)

    def frame(self, timed=False):
        self.rt.set_reuse_weights(self.reuse)
        self.k += 1
        t = self.states[self.k % 2]
        if self.motion:
            self.app.set_triangles(t)
        else:
            self.app.triangles.upload(t)
            self.app.geom.refit()
        if not timed:
            self.app.frame()
            return None
        self.rt.timer_start()
        self.app.frame()
        return self.rt.timer_stop_ms()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "reuse_motion", "reuse_motion.json"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--step", type=float, default=0.05, help="vertical move of the moving triangles, scene units")
    args = ap.parse_args()
    import bench

    tris, cam, workload = bench.load_workload()
    idx = np.arange(len(tris))
    moving = ((idx // 12) % 8 == 0) & ~(tris["emissive"] > 0).any(1)
    up = tris.copy()
    up["vertices"][moving, :, 1] += np.float32(args.step)
    states = (tris, up)
    rt = cedecrt.Runtime(0)  # CRT_MATH_REFERENCE, the default
    result = {"device": rt.device_name(), "nvidia_smi": gpu_info(), "workload": workload, "triangles": int(len(tris)),
              "moving_triangles": int(moving.sum()), "math_mode": "REFERENCE", "step": args.step}
    print(result, flush=True)
    W, H = 3840, 2160
    arms = {name: Animated(rt, states, cam, W, H, reuse, rep, mo) for name, reuse, rep, mo in ARMS}
    for a in arms.values():
        for _ in range(3):
            a.frame()
    rt.sync()
    times = {name: [] for name in arms}
    refit = {name: [] for name in arms}
    for _ in range(args.rounds):
        for name, a in arms.items():
            for _ in range(2):
                a.frame()
            for _ in range(args.frames):
                times[name].append(a.frame(timed=True))
                refit[name].append(a.app.geom.stats()["refit_ms"])
    result["frame_ms_4k"] = {k: {"median": float(np.median(v)), "all": v} for k, v in times.items()}
    result["refit_ms"] = {k: float(np.median(v)) for k, v in refit.items()}
    print("frame ms", {k: v["median"] for k, v in result["frame_ms_4k"].items()}, "refit ms", result["refit_ms"], flush=True)
    km = {}
    for name, a in arms.items():
        a.frame()
        agg = {}
        for _ in range(5):
            a.rt.set_reuse_weights(a.reuse)
            a.k += 1
            t = a.states[a.k % 2]
            if a.motion:
                a.app.set_triangles(t)
            else:
                a.app.triangles.upload(t)
                a.app.geom.refit()
            rt.profile_begin()
            a.app.frame()
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
