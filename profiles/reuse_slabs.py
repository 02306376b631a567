"""Cost of unbiased reuse weights on row slabs (crt_restir_set_halo_surfaces): the halo rows' primary rays and G-buffer
records each slab produces itself.

One GPU command: the fused 10_restir_di frame at 3840x2160 on bench.py's workload (the procedural stand-in when the
blocks_restir cache is absent; the output names the scene), CRT_MATH_REFERENCE, static camera.  Arms, alternated over
several rounds:
  one_slab        slabs.SlabRenderer over the whole image (no halo rows)
  group_2/4/8     slabs.SlabGroup with 2, 4 and 8 slabs of 1080 / 540 / 270 rows on one GPU, linked by plain pointers
                  (direct halo stores): proxies for the slab sizes of 2, 4 and 8 GPUs
each under CRT_REUSE_UNBIASED and, as the floor, CRT_REUSE_REFERENCE (under which the halo work is not issued).
Reports the median frame time (CUDA events on the group's first stream after it has joined the others), the crt_profile
marks summed over the slabs (with slabs sharing the GPU these are stream times, not kernel times), and the kernel times of
the halo raycast and of the halo-surface kernel measured on one context alone (isolated_halo_kernels), with the device's
name and power limit (read-only nvidia-smi query) read in the same run.
Writes JSON (default profiles/reuse_slabs/reuse_slabs.json)."""
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
import slabs  # noqa: E402

MODES = (("unbiased", cedecrt.REUSE_UNBIASED), ("reference", cedecrt.REUSE_REFERENCE))
MATH_NAMES = {cedecrt.MATH_LIBDEVICE: "LIBDEVICE", cedecrt.MATH_EXACT: "EXACT", cedecrt.MATH_FAST: "FAST",
              cedecrt.MATH_REFERENCE: "REFERENCE"}


def isolated_halo_kernels(tris, cam, W, H, frames=5):
    """kernel times of the halo work with nothing else on the GPU: one context renders a slab of 1080 / 540 / 270 rows in
    the middle of the image (both halo bands present) under unbiased weights with halo surfaces, the fused frame on its
    own stream; crt_profile marks averaged over `frames` frames.  Only the kernel times are meant: the slab's halo
    reservoir rows are not exchanged, so its image is not the one a split frame renders."""
    rt = cedecrt.Runtime(0)
    rt.set_math_mode(cedecrt.MATH_REFERENCE)
    rt.set_reuse_weights(cedecrt.REUSE_UNBIASED)
    rt.restir_set_halo_surfaces(True)
    opt = cedecrt.Options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    app = cedecrt.RestirDI(rt, W, H, tris, *cam, opt, fused=True)
    out = {}
    for rows in (H, 1080, 540, 270):
        y0 = (H - rows) // 2 // 8 * 8
        rt.set_row_range(y0, y0 + rows)
        for _ in range(2):
            app.frame()
        rt.sync()
        rt.profile_begin()
        for _ in range(frames):
            app.frame()
        agg = {}
        for name, ms in rt.profile_end():
            agg[name] = agg.get(name, 0.0) + ms / frames
        out["rows_%d" % rows] = {"rows": [y0, y0 + rows], "halo_raycast_ms": round(agg.get("halo_raycast", 0.0), 4),
                                 "halo_surfaces_ms": round(agg.get("halo_surfaces", 0.0), 4),
                                 "raycast_own_rows_ms": round(agg.get("raycast", 0.0), 4)}
    app.geom.destroy()
    rt.close()
    return out


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "reuse_slabs", "reuse_slabs.json"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    args = ap.parse_args()
    import torch

    import bench

    tris, cam, workload = bench.load_workload()
    W, H = args.width, args.height
    torch.cuda.set_device(0)
    torch.cuda.set_stream(torch.cuda.Stream())
    arms = {"one_slab": slabs.SlabRenderer(torch, None, 0, 1, tris, cam, W, H, fused=True)}
    for sub in (2, 4, 8):
        arms["group_%d" % sub] = slabs.SlabGroup(torch, None, 0, 1, tris, cam, W, H, sub=sub)
    for r in arms.values():
        r.set_math_mode(cedecrt.MATH_REFERENCE)
    modes = {s.rt.math_mode for r in arms.values() for s in r.slabs}
    assert len(modes) == 1, modes
    result = {"device": arms["one_slab"].rt.device_name(), "nvidia_smi": gpu_info(), "workload": workload,
              "triangles": int(len(tris)), "math_mode": MATH_NAMES[modes.pop()], "image": [W, H],
              "slab_rows": {k: [b - a for a, b in zip(r.edges, r.edges[1:])] for k, r in arms.items()},
              "multi_gpu": "not measured (one GPU)"}
    print(result, flush=True)

    def run(r, reuse, frames):
        r.set_reuse_weights(reuse)
        for _ in range(frames):
            r.frame()
        r.join()

    for r in arms.values():
        for _, reuse in MODES:
            run(r, reuse, 3)
    torch.cuda.synchronize()
    times = {(k, m): [] for k in arms for m, _ in MODES}
    for _ in range(args.rounds):
        for k, r in arms.items():
            for m, reuse in MODES:
                run(r, reuse, 3)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(r.stream)
                run(r, reuse, args.frames)
                b.record(r.stream)
                b.synchronize()
                times[(k, m)].append(a.elapsed_time(b) / args.frames)
    result["frame_ms"] = {"%s/%s" % key: {"median": float(np.median(v)), "all": v} for key, v in times.items()}
    print("frame ms", {k: round(v["median"], 3) for k, v in result["frame_ms"].items()}, flush=True)
    halo = {}
    for k, r in arms.items():
        for m, reuse in MODES:
            run(r, reuse, 2)
            torch.cuda.synchronize()
            for s in r.slabs:
                s.rt.profile_begin()
            run(r, reuse, 5)
            agg = {}
            for s in r.slabs:
                for name, ms in s.rt.profile_end():
                    agg[name] = agg.get(name, 0.0) + ms / 5
            halo["%s/%s" % (k, m)] = {"halo_raycast_ms": round(agg.get("halo_raycast", 0.0), 4),
                                      "halo_surfaces_ms": round(agg.get("halo_surfaces", 0.0), 4),
                                      "kernels_ms": {n: round(v, 4) for n, v in agg.items()}}
    result["per_frame_summed_over_slabs"] = halo
    result["per_frame_summed_over_slabs_note"] = ("crt_profile marks of slabs that share the GPU: time each slab's stream "
                                                  "spent beside the others' kernels, not kernel time")
    result["halo_kernels_isolated"] = isolated_halo_kernels(tris, cam, W, H)
    print("isolated halo kernels", result["halo_kernels_isolated"], flush=True)
    print("halo ms", {k: (v["halo_raycast_ms"], v["halo_surfaces_ms"]) for k, v in halo.items()}, flush=True)
    for r in arms.values():
        if hasattr(r, "close"):
            r.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1, default=float)
    print(json.dumps(result, default=float)[:3000])


if __name__ == "__main__":
    main()
