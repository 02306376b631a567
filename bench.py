#!/usr/bin/env python
"""bench.py — ReSTIR DI 4K throughput (BASELINE.json metric) on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W]                 this repo's CUDA path
  python bench.py --impl reference ...                                 the reference's own CPU implementation

A "step" is one frame of the reference's frame loop (examples/10_restir_di/10_restir_di.cpp:229-380: raycast,
generate_candidate, temporal_resampling, save_temporal_reservoir, 3 x spatial_resampling, resolve,
tone_mapping) — issued as the fused frame calls of include/cedecrt.h (--mode fused, default; identical images)
or as the reference's launch list (--mode dropin) — over BASELINE config 5: blocks_restir.obj tiled x6 (9 590 208 triangles, 875 892 lights),
3840x2160, temporal + spatial (5 neighbours, r = 30, 3 passes) + visibility reuse, accumulate.

value  = W*H*K / device time of the K frames (CUDA events, max over ranks), buffers resident in HBM —
         the reference's own timing convention (OroStopwatch around the kernel list, 10_restir_di.cpp:254,382).
e2e    = the same loop including, every frame, the device->host copy of the RGBA8 image into pinned host
         memory (10_restir_di.cpp:386-389) — on a copy stream overlapped with the next frame (--readback pipelined,
         default) or copy-then-synchronise like the reference (--readback sync); the per-frame host inputs
         (RayGenerator, eye, Options) travel as kernel parameters.
fast_math = the same K frames with crt_set_math_mode(CRT_MATH_FAST), reported beside the headline (never as it):
         reservoir kernels with fast math, rays and triangle tests exact, radiance 6e-5 from the oracle after 64 frames.
roofline = the dominant kernel by time (a traversal kernel: issue-bound, see DESIGN.md section 4), `traffic` from the
         committed ncu capture; roofline_reservoir_passes = the reservoir kernels' algorithmic bytes / their time.
ref_gpu = the reference's own Orochi/HIPRT CUDA build of 10_restir_di (baseline/_ref/bin/ref_gpu: its unmodified kernel file
         compiled by NVRTC at run time, HIPRT's traversal) on the same GPU, same scene, camera, options and frame count, event-timed
         around the same kernel list (10_restir_di.cpp:254-255,382-383) — run by rank 0 at N = 1 after the timed regions.
frame_hash = after the timed regions: history reset, CRT_MATH_EXACT, frames 1-2 rendered again, the RGBA8 image and the float4
         accumulation hashed row by row (a partition-independent checksum of checksums): the same value at N = 1, 2, 4, 8 and the
         one tests/test_gpu_parity.py::test_bench_frame_hash asserts.
--config 06 | 08 | 09 : BASELINE configs 2-4 (06_ao_hiprt on blocks_ao, 08_nee on blocks_pt, 09_ris with the shadowed target on
         blocks_restir, all 1920x1080) instead of config 5: Mpix/s and Grays/s of the single-kernel frame.
N > 1  : the frame is split into horizontal row slabs, one rank per GPU (strong scaling); scene and BVH are
         replicated; the 87 halo rows of reservoirs the spatial passes read are stored by the producing rank
         directly into its neighbours' buffers over NVLink (--halo p2p, csrc/slab_p2p.cu) or exchanged with
         NCCL send/recv (--halo nccl, and always in --mode dropin).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "cedec-2024-rt_b200", "python"))

W4K, H4K = 3840, 2160
CAM = ((-0.579885, 22.194597, -6.567105), (5.224952, 20.847435, 1.431192))  # 10_restir_di.cpp:188-189


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


# committed `ncu --set full` capture of this command (N = 1, 4K, default mode): newest round first
NCU_SUMMARY = next((q for q in (os.path.join(ROOT, "profiles", "r2", "ncu_r2_summary.csv"),
                                os.path.join(ROOT, "profiles", "r1", "ncu_q_summary.csv")) if os.path.exists(q)), "")
NCU_NAMES = {"raycast": "k_raycast", "candidate_temporal": "k_candidate_temporal", "spatial_fast": "k_spatial_fast",
             "resolve_fast": "k_resolve_fast", "tone_mapping": "k_tone_mapping",
             "trace_visibility_reuse": "k_trace_shadow_queue<2>", "trace_resolve": "k_trace_shadow_queue<1>"}


def _ncu_rows(kernel):
    import csv

    key = NCU_NAMES.get(kernel, kernel)
    if not key or not NCU_SUMMARY:
        return None, None, None
    rows = list(csv.reader(open(NCU_SUMMARY)))
    return rows[0], rows[1], [r for r in rows[2:] if key in r[0]]


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed capture (bytes), or None"""
    h, units, rows = _ncu_rows(kernel)
    if not rows:
        return None
    try:
        ir, iw = h.index("dram__bytes_read.sum"), h.index("dram__bytes_write.sum")
    except ValueError:
        return None
    scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
    vals = [float(r[ir]) * scale.get(units[ir], 1.0) + float(r[iw]) * scale.get(units[iw], 1.0) for r in rows]
    return int(sum(vals) / len(vals)) if vals else None


def ncu_warp_instructions(kernel):
    """smsp__inst_executed.sum per launch of `kernel` from the committed capture (warp instructions), or None"""
    h, units, rows = _ncu_rows(kernel)
    if not rows or "smsp__inst_executed.sum" not in h:
        return None
    i = h.index("smsp__inst_executed.sum")
    vals = [float(r[i]) for r in rows]
    return sum(vals) / len(vals)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index
        self.t0 = self.t1 = None  # timed region (time.time()); samples outside it are dropped when enough lie inside

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        rows = [r for t, r in self.rows if self.t0 is None or (self.t0 <= t <= (self.t1 or t))]
        where = "timed regions"
        if len(rows) < 2:  # nvidia-smi's sampling period can exceed a short timed region: fall back to the whole run
            rows, where = [r for _, r in self.rows], "whole run (warm-up included)"
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "window": where}


def load_workload():
    """BASELINE config 5 scene; falls back to a procedural scene of the same character if the asset cache
    (assets/blocks_restir.tri.xz, staged by oracle/stage_assets.py) is absent, and says so."""
    import scenes

    if scenes.find_scene("blocks_restir"):
        base = scenes.load_scene("blocks_restir")
        return scenes.tile_scene(base, 3, 2, 130.0, 82.0), CAM, "10_restir_di: blocks_restir.obj tiled x6 (3x2, pitch 130/82)"
    tris = scenes.procedural_blocks(n_blocks=800000, seed=1, extent=200.0)
    return tris, ((0.0, 22.0, 0.0), (30.0, 18.0, 30.0)), "10_restir_di: PROCEDURAL stand-in scene (blocks_restir cache not staged)"


# compulsory HBM bytes per pixel of each kernel: (diffuse pixel, sky/emissive pixel).  Per-kernel path: the
# reference struct sizes of SURVEY.md section 8d.  Fused path: what the fused kernels themselves have to move
# (SoA reservoir 72 B, G-buffer 24 B, class 1 B, queue record 64 B) — smaller than the reference-equivalent
# figure, and the one `achieved` is computed from (DESIGN.md section 6).
KERNEL_BYTES = {
    "raycast": (16, 16), "generate_candidate": (92, 92), "temporal_resampling": (244, 16),
    "save_temporal_reservoir": (152, 152), "spatial_resampling": (168, 16), "resolve": (124, 32), "tone_mapping": (20, 20),
    "candidate_temporal": (16 + 72 + 72 + 24 + 1, 16 + 72 + 1), "spatial_fast": (1 + 24 + 72 + 72, 1),
    "resolve_fast": (16 + 1 + 24 + 72 + 64, 16 + 1 + 16),
    "trace_visibility_reuse": (None, None), "trace_resolve": (None, None),  # traversal: per-ray figures below
}
HBM_BOUND = ("temporal_resampling", "save_temporal_reservoir", "spatial_resampling", "tone_mapping", "spatial_fast",
             "candidate_temporal", "resolve_fast")


# ============================================================================================== frame hash
def _row_weights(np, n_words):
    """odd 64-bit multipliers K_i = splitmix64(i) | 1 (numpy uint64 arithmetic wraps modulo 2^64)"""
    with np.errstate(over="ignore"):
        z = (np.arange(n_words, dtype=np.uint64) + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z | np.uint64(1)).view(np.int64)


def frame_hash(torch, dist, r, world, frames=2):
    """Partition-independent fingerprint of the rendered frame, bit-stable across builds: history reset, CRT_MATH_EXACT
    (every operation rounded once in source order, correctly rounded transcendentals — bit-identical to the CPU oracle),
    `frames` frames of the benchmarked loop, then for every image row yi the wrap-around sums
    sum_i word_i * K_i (mod 2^64) over the row's RGBA8 words and over its float4 accumulation words, and FNV-1a-64 over
    those 2 H values in row order.  Every row is hashed by the rank (slab) that rendered it."""
    import numpy as np

    import cedecrt

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    r.join()
    barrier()
    r.set_math_mode(cedecrt.MATH_EXACT)
    r.reset_history()
    barrier()
    for _ in range(frames):
        r.frame()
    r.join()
    barrier()
    first = r.slabs[0]
    W, H = first.W, first.H
    rows = torch.zeros((H, 2), dtype=torch.int64, device="cuda")
    for sl in r.slabs:
        if sl.y1 <= sl.y0:
            continue
        for col, (t, elem) in enumerate(((sl.t_pix, 4), (sl.t_acc, 16))):
            words = sl._rows(t, elem, sl.y0, sl.y1).view(torch.int32).reshape(sl.y1 - sl.y0, -1).to(torch.int64)
            k = torch.from_numpy(_row_weights(np, words.shape[1])).to(words.device)
            h = (words * k).sum(dim=1)  # int64 arithmetic wraps: sums modulo 2^64
            rows[sl.y0:sl.y1, col] = torch.flip(h, dims=[0])  # bottom-up storage: the slab's last row comes first
    if world > 1:
        dist.all_reduce(rows)  # every row was filled by exactly one slab
    data = rows.cpu().numpy().astype("<i8").tobytes()
    h = 0xCBF29CE484222325
    for b in data:
        h = ((h ^ b) * 0x100000001B3) & 0xFFFFFFFFFFFFFFFF
    return {"value": "%016x" % h, "frames": frames, "math": "exact",
            "recipe": "FNV-1a-64 over per-row (RGBA8, accumulation) wrap-around weighted word sums, rows in yi order"}


DUMP_PIXELS = 1 << 20  # pixels sampled by --dump-outputs: 2 x 16 MB of float32 + 8 MB of indices


def dump_outputs(torch, dist, r, rank, out_dir):
    """--dump-outputs DIR: what the last timed frame left for a caller of the frame loop — the RGBA8 image and the float4
    accumulation — at a fixed, seeded sample of DUMP_PIXELS pixel indices (every pixel if the image is smaller), so that two
    builds can be compared output for output.  Written by rank 0 as DIR/pixels.npy (n x 4, float32 of the 0-255 channel
    values), DIR/accumulation.npy (n x 4, float32) and DIR/pixel_index.npy (n, float64: index into the image buffer, whose
    rows are stored bottom-up)."""
    import numpy as np

    torch.cuda.synchronize()
    first = r.slabs[0]
    W, H = first.W, first.H
    acc = torch.zeros(H * W * 4, dtype=torch.int32, device="cuda")  # raw float bits: the sum below only moves them
    pix = torch.zeros(H * W, dtype=torch.int32, device="cuda")
    for sl in r.slabs:  # every row comes from the slab that rendered it
        if sl.y1 <= sl.y0:
            continue
        a, b = (H - sl.y1) * W, (H - sl.y0) * W
        acc[4 * a:4 * b] = sl._rows(sl.t_acc, 16, sl.y0, sl.y1).view(torch.int32)
        pix[a:b] = sl._rows(sl.t_pix, 4, sl.y0, sl.y1).view(torch.int32)
    if dist is not None:
        dist.all_reduce(acc)
        dist.all_reduce(pix)
    if rank != 0:
        return
    n = W * H
    idx = np.arange(n) if n <= DUMP_PIXELS else np.sort(np.random.default_rng(0).choice(n, DUMP_PIXELS, replace=False))
    sel = torch.from_numpy(idx).to("cuda")
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "accumulation.npy"), acc.view(torch.float32).reshape(n, 4)[sel].cpu().numpy())
    np.save(os.path.join(out_dir, "pixels.npy"), pix.view(torch.uint8).reshape(n, 4)[sel].float().cpu().numpy())
    np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))


# ============================================================================================== reference GPU comparator
def run_ref_gpu(W, H, steps, warmup, tiles=(3, 2), timeout=900):
    """the reference's own Orochi/HIPRT CUDA build of examples/10_restir_di on this GPU (baseline/_ref/bin/ref_gpu, built
    by `make -C oracle refgpu` from the reference's sources; see oracle/ref_gpu/ref_gpu_main.cpp): same scene, tiling,
    camera, options and frame count, OroStopwatch around the kernel list like 10_restir_di.cpp:254-255,382-383."""
    import lzma
    import tempfile

    bin_dir = os.path.join(ROOT, "baseline", "_ref", "bin")
    exe = os.path.join(bin_dir, "ref_gpu")
    src = os.path.join(ROOT, "assets", "blocks_restir.tri.xz")
    if not os.path.exists(exe):
        return {"unavailable": "baseline/_ref/bin/ref_gpu not staged (make -C oracle refgpu needs /root/reference)"}
    if not os.path.exists(src):
        return {"unavailable": "assets/blocks_restir.tri.xz not staged"}
    t0 = time.time()
    tmp = tempfile.mkdtemp(prefix="refgpu_")
    tri = os.path.join(tmp, "blocks_restir.tri")
    with lzma.open(src, "rb") as f, open(tri, "wb") as g:
        g.write(f.read())
    env = dict(os.environ)
    env["LD_LIBRARY_PATH"] = bin_dir + ":/usr/local/cuda/lib64:" + env.get("LD_LIBRARY_PATH", "")
    cmd = [exe, "--base", "../", "--tri", tri, "--width", str(W), "--height", str(H), "--tiles-x", str(tiles[0]),
           "--tiles-z", str(tiles[1]), "--frames", str(steps), "--warmup", str(warmup)]
    try:
        pr = subprocess.run(cmd, cwd=bin_dir, env=env, capture_output=True, text=True, timeout=timeout)
    except subprocess.TimeoutExpired:
        return {"unavailable": "timed out after %d s" % timeout}
    finally:
        try:
            os.remove(tri)
            os.rmdir(tmp)
        except OSError:
            pass
    line = [l for l in pr.stdout.splitlines() if l.startswith("{")]
    if not line:
        return {"unavailable": "exit code %d, no result line; stderr tail: %s" % (pr.returncode, pr.stderr[-300:].replace("\n", " | "))}
    out = json.loads(line[-1])
    if "unavailable" in out:
        return {"unavailable": out["unavailable"]}
    return {"value": out["value"], "unit": "Mpix/s", "ms_per_step": out["ms_per_step"], "steps": out["steps"], "warmup": out["warmup"],
            "build_s": out.get("geometry_build_s"), "compile_s": out.get("trace_kernel_compile_s"),
            "mean_radiance": out.get("mean_radiance"), "sky_pixels": out.get("sky_pixels"), "wall_s": round(time.time() - t0, 1),
            "what": "reference Orochi/HIPRT build (HIPRT 2.4 binary, kernels JIT-compiled by NVRTC from the unmodified "
                    "10_restir_di.cu), same GPU, scene, camera, options; CUDA-event time of raycast ... tone_mapping per frame"}


from slabs import HALO as HALO_ROWS, SlabGroup, SlabRenderer  # noqa: E402  (cedec-2024-rt_b200/python/slabs.py)


def dominant_roofline(name, k, hbm_peak, peak_src, issue_peak, sm_mhz, comparable):
    """`roofline` of the JSON line: the dominant kernel by time against the roof that bounds it.  The traversal kernels
    (raycast, trace_*) issue instructions at ~75 % of the schedulers' rate with < 5 % of DRAM bandwidth: their roof is
    instruction issue; the per-pixel reservoir kernels are measured against HBM (roofline_reservoir_passes)."""
    traversal = name in ("raycast", "trace_visibility_reuse", "trace_resolve")
    hbm = {"achieved": k.get("algo_gbs"), "peak": hbm_peak, "unit": "GB/s",
           "frac": round(k["algo_gbs"] / hbm_peak, 4) if k.get("algo_gbs") else None, "peak_source": peak_src}
    out = {"kernel": name, "traffic": ncu_traffic(name) if comparable else None,
           "traffic_source": (os.path.relpath(NCU_SUMMARY, ROOT) + " (dram__bytes_read.sum + dram__bytes_write.sum, one launch)") if NCU_SUMMARY else None}
    if traversal and "issue_frac" in k:
        out.update({"bound": "issue", "achieved": round(k["warp_inst_per_launch"] / (k["ms_per_launch"] * 1e-3) / 1e9, 2),
                    "peak": round(issue_peak / 1e9, 2), "unit": "Gwarp-inst/s", "frac": k["issue_frac"], "hbm": hbm,
                    "note": "dominant kernel by time; a traversal kernel: bound by instruction issue (148 SMs x 4 schedulers x "
                            "%.0f MHz sampled in this run), not by HBM — its algorithmic bytes against the HBM peak are kept under "
                            "`hbm` for reference" % sm_mhz})
    else:
        out.update({"bound": "hbm", **hbm,
                    "note": "dominant kernel by time" + ("; a traversal kernel (issue-bound: see profiles/ for the ncu capture; no "
                            "instruction count for this configuration is committed, so only the HBM figure is given)" if traversal else "")})
    return out


def pixel_classes(torch, renderer):
    """(pixels, diffuse pixels) of this rank's slab(s), from the visibility buffer: a diffuse pixel is one whose
    primary hit is a non-emissive surface — the only pixels with reservoir work and shadow rays."""
    n_px = n_diffuse = 0
    for r in renderer.slabs:
        vis = r._rows(r.t_vis, 16, r.y0, r.y1).view(torch.int32).reshape(-1, 4)[:, 2]
        em = r.t_tris.view(torch.float32).reshape(-1, 15)[:, 12:15]
        is_em = (em > 0).any(1)
        hit = vis >= 0
        diffuse = hit.clone()
        diffuse[hit] = ~is_em[vis[hit].long()]
        n_px += r.W * (r.y1 - r.y0)
        n_diffuse += int(diffuse.sum().item())
    return n_px, n_diffuse


def run_cuda(args):
    # each context drives up to three streams (frame, tail, prefetch) beside torch's and NCCL's: give them hardware queues of
    # their own, so that a kernel of one stream is never queued behind another stream's (the default is 8 connections)
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the CUDA path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    # a real (non-default) torch stream: kernels, copies, NCCL and the timing events all go to it.  (The legacy
    # default stream's handle is 0, which crt_set_stream reads as "use the context's own stream".)
    # high priority: the frame's own kernel sequence is the critical path; the overlapped tail and the prefetched primary rays
    # (the context's second and third streams, default priority) are there to fill what it leaves idle
    stream = torch.cuda.Stream(priority=-1) if args.overlap else torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    # stdout carries exactly one JSON line: whatever libraries print while the run lasts (the image sets
    # NCCL_DEBUG=VERSION, so NCCL writes a version banner to file descriptor 1) goes to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    tris, cam, workload = load_workload()
    W, H = args.width, args.height
    fused = args.mode == "fused"
    # slabs per GPU (--sub; slabs.py: SlabGroup): two slabs on two streams fill each other's ramp-up and drain gaps.  Round 1
    # used two per GPU below 300 rows (+7 % on two GPUs at 272 rows each).  Frame overlap (--overlap, crt_set_frame_overlap)
    # fills the same gaps without coupling two slabs at every spatial pass: on two GPUs at 272 rows each 1329 (neither) /
    # 1413 (two slabs) / 1459 (both) / 1509 Mpix/s (overlap alone) — profiles/r2/tuning.txt.  So one slab per GPU by default.
    sub = args.sub if args.sub > 0 else 1
    if not (fused and args.halo == "p2p" and W % 16 == 0 and H // (world * sub) >= HALO_ROWS + 9):
        sub = 1
    r = None
    if sub > 1:
        r = SlabGroup(torch, dist if world > 1 else None, rank, world, tris, cam, W, H, sub=sub, overlap=bool(args.overlap))
        # pre-flight: two frames; if any slab's wait for a neighbour timed out anywhere, every rank falls back to one slab
        for _ in range(2):
            r.frame()
        torch.cuda.synchronize()
        bad = torch.tensor([0.0], device="cuda")
        try:
            r.check()
        except RuntimeError as e:
            print("bench.py: %s" % e, file=sys.stderr)
            bad += 1
        if world > 1:
            dist.all_reduce(bad)
        if bad.item() > 0:
            r.close()  # unmap the neighbours' buffers ...
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()  # ... on every rank before any rank frees what it exported
            r, sub = None, 1
        else:
            r.reset_history()
            torch.cuda.synchronize()
    if r is None:
        r = SlabRenderer(torch, dist if world > 1 else None, rank, world, tris, cam, W, H, fused=fused, p2p=(args.halo == "p2p"),
                         overlap=bool(args.overlap))
    import cedecrt
    math_mode = {"reference": cedecrt.MATH_REFERENCE, "libdevice": cedecrt.MATH_LIBDEVICE, "fast": cedecrt.MATH_FAST,
                 "exact": cedecrt.MATH_EXACT}[args.math]
    r.set_math_mode(math_mode)
    stats = r.geom.stats()
    sm_count = torch.cuda.get_device_properties(local).multi_processor_count
    if world * sub > 1 and not args.no_balance:
        r.calibrate(rounds=3, frames=4)  # static camera: balance the slab heights on throw-away frames before the sequence starts

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        r.frame()
    barrier()
    launches0 = r.launch_count()
    rays0 = r.shadow_rays_traced()
    decided0 = r.rays_decided_at_emission()[0]
    sampler.mark_begin()
    # ---- timed: K frames, resident buffers
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        r.frame()
    r.join()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs:
        dump_outputs(torch, dist if world > 1 else None, r, rank, args.dump_outputs)
    launches = r.launch_count() - launches0
    rays1 = r.shadow_rays_traced()
    shadow_rays = [(b - a) / args.steps for a, b in zip(rays0, rays1)]  # per frame: (visibility reuse, resolve)
    decided_vr = (r.rays_decided_at_emission()[0] - decided0) / args.steps  # this rank's, settled by the own-triangle pre-test
    # ---- timed: K frames end to end (per-frame D2H of the RGBA8 image into pinned host memory)
    if args.readback == "pipelined":
        r.wait_download(r.download_pixels_async())  # allocates the copy stream and the pinned images, untimed
    barrier()
    t_e0, t_e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_e0.record()
    if args.readback == "sync":
        for _ in range(args.steps):
            r.frame()
            r.download_pixels()
            for sl in r.slabs:
                sl.stream.synchronize()  # oroStreamSynchronize after the copy (10_restir_di.cpp:389)
    else:
        # pipelined: frame i's image travels on a copy stream while frame i+1 renders; the host takes delivery of
        # image i-1 (one frame of latency, as a display loop has); every frame's copy lies inside the timed region
        prev = None
        for _ in range(args.steps):
            r.frame()
            slot = r.download_pixels_async()
            if prev is not None:
                r.wait_download(prev)
            prev = slot
        r.wait_download(prev)
        for ev in r.last_copy_events(prev):
            torch.cuda.current_stream().wait_event(ev)
    r.join()
    t_e1.record()
    barrier()
    ms_e2e = t_e0.elapsed_time(t_e1)
    # ---- the two timed regions together can be shorter than nvidia-smi's sampling period (8 frames at N = 8 take
    # 16 ms): keep the same frames running, untimed, until the sampled window under load is about 1.5 s long
    n_probe = torch.tensor([max(0, int((1.5 - (time.time() - sampler.t0)) / max(ms / args.steps / 1e3, 1e-4)))],
                           dtype=torch.int64, device="cuda")
    if world > 1:
        dist.broadcast(n_probe, 0)
    for _ in range(min(int(n_probe.item()), 5000)):
        r.frame()
    barrier()
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "%s + %d more frames of the same loop (untimed), %.2f s under load" % (
            clocks.get("window", "timed regions"), int(n_probe.item()), sampler.t1 - sampler.t0)
    # ---- the same K frames in CRT_MATH_FAST (reported next to the headline, never as the headline: its radiance is
    # inside the north star's tolerance of the oracle but not bit-comparable; include/cedecrt.h)
    ms_fast = None
    if fused and args.math in ("reference", "libdevice") and not args.no_fast_line:
        r.set_math_mode(cedecrt.MATH_FAST)
        for _ in range(2):
            r.frame()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            r.frame()
        r.join()
        f1.record()
        barrier()
        ms_fast = f0.elapsed_time(f1)
        r.set_math_mode(math_mode)
        r.frame()
    # ---- per-kernel device times: an event after every launch (crt_profile_begin/end), steady-state frames
    n_prof = max(2, min(args.steps, 4))
    r.halo_bytes = 0
    r.rt.profile_begin()
    for _ in range(n_prof):
        r.frame()
    marks = r.rt.profile_end()
    halo_bytes_per_frame = r.halo_bytes // n_prof
    per_kernel = {}
    for name, t_ms in marks:
        per_kernel.setdefault(name, []).append(t_ms)
    timed_out = 0.0  # a halo wait that gave up (k_signal_wait's watchdog) invalidates every number of this run
    try:
        r.check()
    except RuntimeError as e:
        print("bench.py: %s" % e, file=sys.stderr)
        timed_out = 1.0
    n_px, n_diffuse = pixel_classes(torch, r)
    fhash = None
    if not args.no_frame_hash:
        fhash = frame_hash(torch, dist if world > 1 else None, r, world)
        r.set_math_mode(math_mode)
    # rays actually traced per frame: 1 primary per pixel + the shadow rays counted by the tracer (the reference traces
    # 2 per diffuse pixel; the fused frame skips those whose answer it already holds, see include/cedecrt.h)
    rays = n_px + sum(shadow_rays)

    own_ms = sum(t_ms for name, t_ms in marks if name != "signal_wait") / n_prof  # this slab's kernels, waiting excluded
    slab_ms = torch.zeros(world, dtype=torch.float64, device="cuda")
    slab_ms[rank] = own_ms
    if world > 1:
        dist.all_reduce(slab_ms)
    t = torch.tensor([ms, ms_e2e, float(rays), float(shadow_rays[0]), float(shadow_rays[1]), float(n_px), float(n_diffuse),
                      float(ms_fast or 0.0), timed_out], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms, ms_e2e, rays = tmax[0].item(), tmax[1].item(), tsum[2].item()
        ms_fast = tmax[7].item() if ms_fast is not None else None
    rays_vr, rays_rs, all_px, all_diffuse = (t[3].item(), t[4].item(), t[5].item(), t[6].item()) if world == 1 else \
        (tsum[3].item(), tsum[4].item(), tsum[5].item(), tsum[6].item())
    any_timed_out = (t[8].item() if world == 1 else tsum[8].item()) > 0
    if rank == 0:
        n_img = W * H
        peak, peak_src = measured_peaks()
        kern = {}
        for name, ts in per_kernel.items():
            per_launch = sum(ts) / len(ts)
            bd, bs = KERNEL_BYTES.get(name, (None, None))
            k = {"ms_per_launch": round(per_launch, 4), "launches_per_frame": round(len(ts) / n_prof, 2)}
            if bd is not None:
                nbytes = bd * n_diffuse + bs * (n_px - n_diffuse)
                k["algo_bytes_per_launch"] = int(nbytes)
                k["algo_gbs"] = round(nbytes / per_launch / 1e6, 1)
            elif name == "trace_resolve":
                k["algo_bytes_per_launch"] = int(96 * shadow_rays[1])  # R 64 B record, RMW float4 accumulation
                k["algo_gbs"] = round(96 * shadow_rays[1] / per_launch / 1e6, 1)
                k["mrays_per_s"] = round(shadow_rays[1] / per_launch / 1e3, 1)
            elif name == "trace_visibility_reuse":
                k["mrays_per_s"] = round(shadow_rays[0] / per_launch / 1e3, 1)
            kern[name] = k
        # instruction-issue roofline: warp instructions per launch (committed ncu capture of this command: they do not
        # depend on the clock) / the live launch time, against SMs x 4 schedulers x the SM clock sampled during this run
        sm_mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0
        issue_peak = sm_count * 4 * sm_mhz * 1e6  # warp instructions per second
        comparable = world == 1 and fused and (W, H) == (W4K, H4K) and args.math == "reference"
        for name, k in kern.items():
            inst = ncu_warp_instructions(name) if comparable else None
            if inst:
                k["warp_inst_per_launch"] = int(inst)
                # (clamped: for a 0.1 ms kernel the event-to-event time of the profile pass can come out a little shorter
                # than its instructions allow at the sampled clock)
                k["issue_frac"] = min(1.0, round(inst / (k["ms_per_launch"] * 1e-3) / issue_peak, 4))
        # k_candidate_temporal against the roof that bounds it (DESIGN.md section 4): one L1 wavefront per lane and 256-bit
        # load of its 32 random 64-byte light records (every lane its own 128-byte line), one wavefront per SM and clock
        if "candidate_temporal" in kern and world == 1:
            k = kern["candidate_temporal"]
            wavefronts = n_diffuse * 32 * 2
            k["l1_wavefronts_per_launch"] = int(wavefronts)
            k["l1_wavefront_frac"] = round(wavefronts / sm_count / (sm_mhz * 1e6) / (k["ms_per_launch"] * 1e-3), 4)
        frame_ms_by_kernel = {k: v["ms_per_launch"] * v["launches_per_frame"] for k, v in kern.items()}
        dominant = max(frame_ms_by_kernel, key=frame_ms_by_kernel.get)
        passes = [k for k in kern if k in HBM_BOUND]
        res_bytes = sum(kern[k]["algo_bytes_per_launch"] * kern[k]["launches_per_frame"] for k in passes)
        res_ms = sum(frame_ms_by_kernel[k] for k in passes)
        dom = kern[dominant]
        out = {
            "metric": "ReSTIR DI 4K Mpix/s", "value": round(n_img * args.steps / ms / 1e3, 3), "unit": "Mpix/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "width": W, "height": H, "triangles": r.n_tris, "lights": r.n_lights,
                       "options": "temporal+spatial(5 nbrs, r=30, 3 passes)+visibility reuse, accumulate, ris 32",
                       "camera": "10_restir_di.cpp:188-189",
                       "mode": "fused frame (crt_restir_frame_begin / spatial_pass / frame_end, SoA reservoirs)" if fused
                               else "per-kernel launch list (drop-in, AoS reservoirs)",
                       "frame_overlap": ("tail of frame f (resolve rays, tone mapping) on a second stream beside the head of frame f+1"
                                         if getattr(r.slabs[0], "overlap", False) else "none: frames strictly serial"),
                       "slab_edges": r.edges,
                       "partition": "%d row slab(s)%s, halo %d rows, %s" % (
                           world * sub, " (%d per GPU, one CUDA stream each)" % sub if sub > 1 else "", HALO_ROWS, "halo rows stored directly into the neighbours' buffers over NVLink "
                           "(cudaIpc peer pointers, csrc/slab_p2p.cu)" if r.p2p else
                           "%d halo bytes sent per frame by rank 0 (NCCL send/recv)" % halo_bytes_per_frame),
                       "l2": "per-frame working set (3 x 600 MB reservoir buffers) exceeds the 126 MB L2; no flush needed",
                       "math": {"reference": "CRT_MATH_REFERENCE: FMA contraction, IEEE division / square root, libdevice functions (nvcc / NVRTC "
                                             "defaults: the reference's own GPU arithmetic); traversal and triangle tests uncontracted",
                                "libdevice": "libdevice float functions, -fmad=false, IEEE division (bit-faithful to the CPU oracle's arithmetic)",
                                "exact": "correctly rounded transcendentals, -fmad=false (bit-identical to the CPU oracle)",
                                "fast": "CRT_MATH_FAST: reservoir kernels with FMA contraction, approximate division and hardware "
                                        "transcendentals; traversal and triangle tests exact; radiance within the north star's "
                                        "tolerance of the oracle (tests/test_gpu_parity.py)"}[args.math]},
            "grays_per_s": round(rays * args.steps / ms / 1e6, 4), "rays_per_frame": int(rays),
            "rays": {"primary": int(all_px), "visibility_reuse": int(rays_vr), "resolve": int(rays_rs),
                     "reference_would_trace": int(all_px + 2 * all_diffuse),
                     "visibility_reuse_decided_at_emission_rank0": int(decided_vr),
                     "note": "per frame, counted by the tracer (crt_shadow_rays_traced); the reference traces one "
                             "visibility-reuse and one resolve ray per diffuse pixel, the fused frame omits those "
                             "whose outcome cannot be read (candidate lost the temporal merge) or is already known "
                             "(resolve ray identical to a traced visibility-reuse ray), and settles a visibility-reuse "
                             "ray without a walk when the triangle it starts on stops it (crt_rays_decided_at_emission; "
                             "not counted in grays_per_s)"},
            "e2e": {"value": round(n_img * args.steps / ms_e2e / 1e3, 3), "unit": "Mpix/s",
                    "h2d_bytes_per_step": 96, "d2h_bytes_per_step": 4 * n_img,
                    "readback": args.readback,
                    "note": "per-frame inputs (RayGenerator 36 B, eye 12 B, Options 48 B) go as kernel parameters; "
                            "the RGBA8 frame is copied to pinned host memory every step" + (
                                " on a copy stream, overlapped with the next frame (SlabRenderer.download_pixels_async)"
                                if args.readback == "pipelined" else
                                " on the frame's stream, followed by a stream synchronise (10_restir_di.cpp:386-389)")},
            "fast_math": None if not ms_fast else {
                "value": round(n_img * args.steps / ms_fast / 1e3, 3), "unit": "Mpix/s", "ms_per_step": round(ms_fast / args.steps, 4),
                "note": "same frames with crt_set_math_mode(CRT_MATH_FAST): reservoir kernels with FMA contraction, approximate "
                        "division and hardware transcendentals, rays and triangle tests exact; mean relative L1 against the "
                        "oracle after 64 frames 6e-5 (tolerance 1e-3; profiles/r1/long_horizon_parity.txt, "
                        "tests/test_gpu_parity.py::test_fast_math_mode_within_tolerance_over_64_frames). Not the headline."},
            "gpu_launches": int(launches),
            "halo_wait_timed_out": bool(any_timed_out),  # true = a slab gave up waiting for a neighbour: the run is invalid
            "clocks": clocks,
            "roofline": dominant_roofline(dominant, dom, peak, peak_src, issue_peak, sm_mhz, comparable),
            "roofline_issue": {"peak_warp_inst_per_s": issue_peak, "sm_count": sm_count, "schedulers_per_sm": 4, "sm_mhz": sm_mhz,
                               "frame_frac": round(sum(k["warp_inst_per_launch"] * k["launches_per_frame"] for k in kern.values()
                                                       if "warp_inst_per_launch" in k) / (ms / args.steps * 1e-3) / issue_peak, 4)
                               if comparable and any("warp_inst_per_launch" in k for k in kern.values()) else None,
                               "source": os.path.relpath(NCU_SUMMARY, ROOT) if NCU_SUMMARY else None,
                               "note": "per kernel: kernels[*].issue_frac = smsp__inst_executed.sum of the committed ncu capture / "
                                       "live launch time / (SMs x 4 x sampled SM clock)"},
            "roofline_reservoir_passes": {"bound": "hbm", "achieved": round(res_bytes / res_ms / 1e6, 1), "peak": peak,
                                          "unit": "GB/s", "frac": round(res_bytes / res_ms / 1e6 / peak, 4),
                                          "kernels": passes, "ms_per_frame": round(res_ms, 4)},
            "kernels": kern,
            "pixels": {"slab": n_px, "diffuse": n_diffuse},
            "slab_kernel_ms": [round(x, 4) for x in slab_ms.tolist()],  # per rank: sum of its own kernels per frame
            "bvh": {k: stats[k] for k in ("n_nodes", "max_depth", "build_ms", "node_bytes", "tri_bytes")},
            "frame_hash": fhash,
        }
        if world == 1 and not args.no_ref_gpu and (W, H) == (W4K, H4K):
            torch.cuda.synchronize()
            out["ref_gpu"] = run_ref_gpu(W, H, args.steps, args.warmup)
            if "value" in out["ref_gpu"]:
                out["ref_gpu"]["vs_ours"] = round(out["value"] / out["ref_gpu"]["value"], 3)
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline_sample(r, tris, cam, W, H, rows=args.cpu_rows)
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()



# ============================================================================================== BASELINE configs 2-4
EXAMPLES = {
    # 06_ao_hiprt.cpp:95,115 + misc.hpp:217-218 camera; N_Rays as BASELINE config 2 asks (the reference hard-codes 64)
    "06": dict(scene="blocks_ao", cam=((8.0, 8.0, 8.0), (0.0, 0.0, 0.0)), ao_rays=32, kernel="ao_06", ncu="k_ao",
               workload="06_ao_hiprt: blocks_ao.obj, 1920x1080, 32 AO rays per hit pixel (pure any-hit traversal)"),
    # 08_nee.cpp:135-140 camera; max depth 4, accumulate (BASELINE config 3)
    "08": dict(scene="blocks_pt", cam=((5.983407, 13.970583, -28.553869), (-5.354514, 4.815835, -2.047728)), kernel="path_trace_08",
               ncu="k_path_trace<8", options=dict(accumulate=1, max_depth=4),
               workload="08_nee: blocks_pt.obj, 1920x1080, 1 spp per frame, max depth 4, accumulating"),
    # 09_ris.cpp:149-154 camera; 32 candidates with visibility inside the target function (BASELINE config 4)
    "09": dict(scene="blocks_restir", cam=CAM, kernel="path_trace_09", ncu="k_path_trace<9",
               options=dict(accumulate=1, max_depth=6, ris_sample_count=32, use_shadowed_target_function=1),
               workload="09_ris: blocks_restir.obj, 1920x1080, 32 light candidates per vertex, shadowed target function, max depth 6"),
}


def run_example(args):
    """--config 06 | 08 | 09: the single-kernel frames of examples 06-09 (kernel + tone mapping for 08/09, as their host
    loops launch them) at 1920x1080 on the example's own scene and camera.  N > 1: row slabs, no exchange (every pixel
    is independent).  Rays are counted by the kernels themselves (crt_inline_rays_traced)."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import cedecrt
    import scenes

    ex = EXAMPLES[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the CUDA path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W, H = (1920, 1080) if (args.width, args.height) == (W4K, H4K) else (args.width, args.height)
    tris = scenes.load_scene(ex["scene"])
    math_mode = {"reference": cedecrt.MATH_LIBDEVICE, "libdevice": cedecrt.MATH_LIBDEVICE, "fast": cedecrt.MATH_LIBDEVICE,
                 "exact": cedecrt.MATH_EXACT}[args.math]  # the per-kernel entry points know LIBDEVICE and EXACT
    rt = cedecrt.Runtime(local, math_mode)
    rt.set_stream(stream.cuda_stream)
    from slabs import slab_rows
    y0, y1 = slab_rows(H, world, rank)
    rt.set_row_range(y0, y1)
    d_tris = rt.to_device(tris)
    lights = cedecrt.light_indices(tris)
    d_lights = rt.to_device(lights) if len(lights) else None  # blocks_ao has no emissive triangle; 06 takes no light list
    geom = rt.build_geometry(d_tris)
    stats = geom.stats()
    raygen = cedecrt.lookat(ex["cam"][0], ex["cam"][1], W, H)
    n = W * H
    pixels = rt.buffer(np.uint8, 4 * n)
    accum = rt.buffer(cedecrt.FLOAT4, n)
    rt.clear(accum, W, H)
    opt = cedecrt.Options(**ex.get("options", {}))
    host = torch.empty(4 * W * max(y1 - y0, 1), dtype=torch.uint8).pin_memory()
    t_pix = torch.as_tensor(__import__("slabs").CudaArrayView(pixels.ptr, 4 * n), device=torch.device("cuda", local))
    state = {"frame": 0}

    def frame():
        state["frame"] += 1
        if args.config == "06":
            rt.ao(pixels, raygen, W, H, geom, d_tris, ex["ao_rays"])
        else:
            rt.path_trace(int(args.config), W, H, state["frame"], geom, d_tris, d_lights, raygen, opt, accum)
            rt.tone_mapping(pixels, accum, W, H)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        frame()
    barrier()
    launches0, rays0 = rt.launch_count(), rt.inline_rays_traced()
    decided0 = rt.rays_decided_at_emission()[1]
    sampler.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        frame()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches, rays1 = rt.launch_count() - launches0, rt.inline_rays_traced()
    rays = [(b - a) / args.steps for a, b in zip(rays0, rays1)]
    decided = (rt.rays_decided_at_emission()[1] - decided0) / args.steps
    # end to end: the frame plus the device -> host copy of this rank's RGBA8 rows and a stream synchronise
    # (06_ao_hiprt.cpp / 08_nee.cpp / 09_ris.cpp read back and display every frame)
    rows_px = t_pix[(H - y1) * W * 4:(H - y0) * W * 4]
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        frame()
        host[:rows_px.numel()].copy_(rows_px, non_blocking=True)
        stream.synchronize()
    t1.record()
    barrier()
    ms_e2e = t0.elapsed_time(t1)
    n_probe = max(0, int((1.5 - (time.time() - sampler.t0)) / max(ms / args.steps / 1e3, 1e-4)))
    for _ in range(min(n_probe, 2000)):
        frame()
    barrier()
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    rt.profile_begin()
    for _ in range(2):
        frame()
    marks = rt.profile_end()
    t = torch.tensor([ms, ms_e2e, rays[0], rays[1]], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax, tsum = t.clone(), t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms, ms_e2e, rays = tmax[0].item(), tmax[1].item(), [tsum[2].item(), tsum[3].item()]
    if rank == 0:
        per = {}
        for name, t_ms in marks:
            per.setdefault(name, []).append(t_ms)
        kern = {k: {"ms_per_launch": round(sum(v) / len(v), 4), "launches_per_frame": len(v) / 2, "ms_per_frame": round(sum(v) / 2, 4)}
                for k, v in per.items()}
        sm_count = torch.cuda.get_device_properties(local).multi_processor_count
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        issue_peak = sm_count * 4 * sm_mhz * 1e6
        main_name = max(kern, key=lambda k: kern[k]["ms_per_frame"])  # the dominant kernel of the frame
        ncu_name = {"ao_emit": "k_ao_emit", "trace_ao": "k_trace_shadow_queue<3>", "ao_finish": "k_ao_finish", "ao_06": "k_ao<",
                    "path_trace": ex["ncu"], "trace_shadow": "k_trace_shadow_queue<4>", "pt_closest": "k_pt_closest",
                    "pt_vertex": "k_pt_vertex", "pt_replay": "k_pt_replay", "pt_shade_bounce": "k_pt_shade_bounce"}.get(main_name, main_name)
        inst = ncu_warp_instructions(ncu_name) if world == 1 and (W, H) == (1920, 1080) else None
        roof = {"kernel": main_name, "bound": "issue", "unit": "Gwarp-inst/s", "peak": round(issue_peak / 1e9, 2),
                "achieved": None, "frac": None, "traffic": None,
                "note": "the frame's dominant kernel, a traversal kernel: bound by instruction issue, not HBM (DRAM throughput of the committed ncu capture "
                        "is a few percent of peak); warp instructions from the committed capture / live kernel time"}
        if inst and main_name in kern:
            roof["achieved"] = round(inst / (kern[main_name]["ms_per_launch"] * 1e-3) / 1e9, 2)
            roof["frac"] = round(inst / (kern[main_name]["ms_per_launch"] * 1e-3) / issue_peak, 4)
            roof["traffic"] = ncu_traffic(ncu_name)
        out = {
            "metric": "%s 1080p Mpix/s" % ex["kernel"], "value": round(n * args.steps / ms / 1e3, 3), "unit": "Mpix/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": ex["workload"], "width": W, "height": H, "triangles": int(len(tris)), "lights": int(len(lights)),
                       "partition": "%d row slab(s), no exchange" % world,
                       "l2": "one launch per frame over the whole image; scene + BVH (%d MB) exceed nothing: L2-resident for "
                             "blocks_ao, larger than L2 for blocks_pt / blocks_restir" % ((stats["node_bytes"] + stats["tri_bytes"]) // 2**20),
                       "math": "libdevice functions, uncontracted arithmetic (the per-kernel entry points' default)"},
            "grays_per_s": round(sum(rays) * args.steps / ms / 1e6, 4), "rays_per_frame": int(sum(rays)),
            "rays": {"closest_hit": int(rays[0]), "shadow_or_ao": int(rays[1]), "shadow_decided_at_emission": int(decided),
                     "note": "per frame, counted by the kernel itself (crt_inline_rays_traced), SURVEY.md section 8d accounting; "
                             "shadow rays that the triangle they start on stops are settled by the emitting kernel without a walk "
                             "(crt_rays_decided_at_emission) and are not counted in grays_per_s"},
            "e2e": {"value": round(n * args.steps / ms_e2e / 1e3, 3), "unit": "Mpix/s", "h2d_bytes_per_step": 132,
                    "d2h_bytes_per_step": 4 * n, "note": "frame + RGBA8 device->host copy into pinned memory + stream synchronise"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "kernels": kern,
            "bvh": {k: stats[k] for k in ("n_nodes", "max_depth", "build_ms", "node_bytes", "tri_bytes")},
        }
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_example_sample(args.config, ex, tris, W, H)
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def cpu_example_sample(config, ex, tris, W, H, rows=16):
    """cpu_baseline for --config 06/08/09: the reference's own kernel as host C++ (oracle/_ref/libref_NN.so, else the
    port) on a band of `rows` image rows of frame 1, all host threads"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np

    import orc

    kind = "reference" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_%s.so" % config)) else "port"
    o = orc.load(kind, int(config))
    o.set_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    if kind == "port":
        o.set_example(int(config))
    g = o.geom_build(tris)
    rg = o.lookat(ex["cam"][0], ex["cam"][1], W, H)
    y0 = (H - rows) // 2
    o.set_range(y0 * W, (y0 + rows) * W)
    t0 = time.perf_counter()
    if config == "06":
        if kind == "reference":
            n_rays = 64  # hard-coded in the reference kernel (06_ao_hiprt.cu:71)
        else:
            n_rays = ex["ao_rays"]
        o.ao(W, H, g, tris, rg, n_rays)
        what = "%d AO rays per hit pixel%s" % (n_rays, " (the reference kernel's hard-coded count; the CUDA arm traces 32)" if n_rays != ex["ao_rays"] else "")
    else:
        opt = orc.make_options(**ex.get("options", {}))
        o.path_trace(W, H, 1, g, tris, orc.light_indices(tris), rg, opt, np.zeros((W * H, 4), np.float32))
        what = "one path_trace launch"
    sec = time.perf_counter() - t0
    o.set_range(0, -1)
    return {"value": round(rows * W / sec / 1e6, 4), "unit": "Mpix/s", "cores": o.threads(), "kind": kind, "seconds": round(sec, 3),
            "sample": "frame 1, image rows %d..%d of the %dx%d frame (%d px), %s; BVH build excluded" % (y0, y0 + rows, W, H, rows * W, what)}

# ============================================================================================== CPU arms
def cpu_band_run(o, tris, cam, W, H, rows, frames, bufs=None):
    """one bounded sample of the workload on the CPU oracle: every kernel of the frame loop restricted to a
    band of `rows` image rows (orc_set_range); full-size zero-initialised buffers.  Returns seconds per kernel."""
    import numpy as np

    import orc

    y0 = (H - rows) // 2
    o.set_range(y0 * W, (y0 + rows) * W)
    opt = orc.make_options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
    n = W * H
    if bufs is None:
        bufs = dict(vis=np.zeros(n, orc.VISIBILITY), r0=np.zeros(n, orc.RESERVOIR), r1=np.zeros(n, orc.RESERVOIR),
                    tmp=np.zeros(n, orc.RESERVOIR), acc=np.zeros((n, 4), np.float32), pix=np.zeros(4 * n, np.uint8))
        bufs["vis"]["index"] = -1
    g = bufs.get("geom") or o.geom_build(tris)
    bufs["geom"] = g
    rg = o.lookat(cam[0], cam[1], W, H)
    lights = orc.light_indices(tris)
    eye = np.asarray(cam[0], np.float32)
    times = {}

    def run(name, fn, *a):
        t0 = time.perf_counter()
        fn(*a)
        times[name] = times.get(name, 0.0) + time.perf_counter() - t0

    for f in frames:
        run("raycast", o.raycast, W, H, g, tris, rg, bufs["vis"])
        run("generate_candidate", o.generate_candidate, W, H, f, g, tris, bufs["vis"], eye, lights, opt, bufs["r0"])
        run("temporal_resampling", o.temporal_resampling, W, H, f, g, tris, bufs["vis"], eye, opt, bufs["tmp"], bufs["r0"])
        run("save_temporal_reservoir", o.save_temporal_reservoir, W, H, bufs["r0"], bufs["tmp"])
        bi, bo = bufs["r0"], bufs["r1"]
        for k in range(3):
            if k:
                bi, bo = bo, bi
            run("spatial_resampling", o.spatial_resampling, W, H, f, k, g, tris, bufs["vis"], eye, opt, bi, bo)
        run("resolve", o.resolve, bufs["acc"], W, H, g, tris, bufs["vis"], eye, opt, bo)
        run("tone_mapping", o.tone_mapping, bufs["acc"], W, H, bufs["pix"])
    o.set_range(0, -1)
    return times, bufs


def load_cpu_oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import orc

    if orc.have_reference():
        return orc.load("reference", 10), "reference"
    return orc.load("port"), "port"


def cpu_baseline_sample(r, tris, cam, W, H, rows=64):
    """cpu_baseline of the CUDA arm's JSON line: the reference's CPU implementation timed on this box's host cores
    on a bounded sample (a band of rows of the same frame)."""
    o, kind = load_cpu_oracle()
    o.set_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    times, _ = cpu_band_run(o, tris, cam, W, H, rows, frames=[1])
    sec = sum(times.values())
    return {"value": round(rows * W / sec / 1e6, 4), "unit": "Mpix/s", "cores": o.threads(), "kind": kind,
            "sample": "frame 1, image rows %d..%d of the %dx%d frame (%d px), all 9 kernel launches of the frame loop, "
                      "OpenMP over pixels; BVH build excluded" % ((H - rows) // 2, (H - rows) // 2 + rows, W, H, rows * W),
            "seconds": round(sec, 3), "seconds_by_kernel": {k: round(v, 3) for k, v in times.items()}}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref: its unmodified kernels as
    host C++ with OpenMP; else the port), all host threads, same config; each step = one frame of a bounded band."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    o, kind = load_cpu_oracle()
    # torch.distributed.run exports OMP_NUM_THREADS=1 to its workers: ask for every host thread explicitly
    o.set_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    tris, cam, workload = load_workload()
    W, H, rows = args.width, args.height, args.cpu_rows
    bufs = None
    frame = 0
    for _ in range(args.warmup):
        frame += 1
        _, bufs = cpu_band_run(o, tris, cam, W, H, rows, [frame], bufs)
    t0 = time.perf_counter()
    per_kernel = {}
    for _ in range(args.steps):
        frame += 1
        times, bufs = cpu_band_run(o, tris, cam, W, H, rows, [frame], bufs)
        for k, v in times.items():
            per_kernel[k] = per_kernel.get(k, 0.0) + v
    sec = sum(per_kernel.values())
    wall = time.perf_counter() - t0
    value = round(rows * W * args.steps / sec / 1e6, 4)
    sample = ("each step = one frame over image rows %d..%d of the %dx%d frame (%d px), all kernels of the frame loop; "
              "BVH build excluded" % ((H - rows) // 2, (H - rows) // 2 + rows, W, H, rows * W))
    print(json.dumps({
        "impl": "reference", "metric": "ReSTIR DI 4K Mpix/s", "value": value, "unit": "Mpix/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(sec / args.steps * 1e3, 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "width": W, "height": H, "triangles": int(len(tris)),
                   "options": "temporal+spatial(5 nbrs, r=30, 3 passes)+visibility reuse, accumulate, ris 32",
                   "sample": sample},
        "cpu_baseline": {"value": value, "unit": "Mpix/s", "cores": o.threads(), "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": round(wall, 2),
        "seconds_by_kernel": {k: round(v, 3) for k, v in per_kernel.items()},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--width", type=int, default=W4K)
    ap.add_argument("--height", type=int, default=H4K)
    ap.add_argument("--cpu-rows", type=int, default=192, help="band height of the CPU arm's per-step sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fast-line", action="store_true", help="skip the additional CRT_MATH_FAST measurement")
    ap.add_argument("--sub", type=int, default=0,
                    help="row slabs (contexts + streams) per GPU (slabs.py: SlabGroup); default 1")
    ap.add_argument("--no-balance", action="store_true", help="N > 1: keep equal-height slabs (no calibration frames)")
    ap.add_argument("--halo", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1, fused mode: halo rows by direct peer stores (default) or NCCL send/recv")
    ap.add_argument("--math", default="reference", choices=["reference", "libdevice", "fast", "exact"],
                    help="arithmetic of the reservoir kernels (include/cedecrt.h: CRT_MATH_*); reference = nvcc/NVRTC defaults, "
                         "the reference's own GPU arithmetic")
    ap.add_argument("--overlap", type=int, default=1, choices=[0, 1],
                    help="1 (default): the frame's tail (resolve rays + tone mapping) runs on a second stream beside the next "
                         "frame's raycast / candidate kernels (crt_set_frame_overlap); 0: strictly serial frames like the reference")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip the reference Orochi/HIPRT comparator run (N = 1, 4K)")
    ap.add_argument("--no-frame-hash", action="store_true", help="skip the exact-mode frame fingerprint")
    ap.add_argument("--config", default="10", choices=["10", "06", "08", "09"],
                    help="10: BASELINE config 5 (default); 06 / 08 / 09: configs 2-4 at 1920x1080 (single-kernel frames)")
    ap.add_argument("--readback", default="pipelined", choices=["pipelined", "sync"],
                    help="e2e: overlap each frame's device->host copy with the next frame (default) or copy and "
                         "synchronise after every frame like the reference's loop")
    ap.add_argument("--mode", default="fused", choices=["fused", "dropin"],
                    help="fused: one crt_restir_* frame call sequence (default); dropin: the reference's launch list")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed frames, write the last one's RGBA8 image and accumulation (a seeded sample of "
                         "pixels) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "cuda" or args.config != "10"):
        ap.error("--dump-outputs is available for the default workload (--impl cuda --config 10)")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        if args.config != "10":
            run_example(args)
        else:
            run_cuda(args)


if __name__ == "__main__":
    main()
