"""TEST INFRASTRUCTURE — one rank of the multi-GPU row-slab test under unbiased reuse weights
(tests/test_gpu_reuse_slabs.py::test_unbiased_slabs_on_gpus, torch.distributed.run, NCCL).  Every rank renders its slab
(slabs.SlabRenderer / SlabGroup, the objects bench.py times) and, on the same GPU, the whole frame as a single slab, both
with CRT_REUSE_UNBIASED and a camera that moves twice; its rows must be identical."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in ("oracle", "tests", os.path.join("cedec-2024-rt_b200", "python")):
    sys.path.insert(0, os.path.join(ROOT, p))
import cedecrt  # noqa: E402
import slabs  # noqa: E402
from helpers import small_scene  # noqa: E402


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    torch.cuda.set_stream(torch.cuda.Stream())
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    # fused (direct peer stores) | fused_nccl | group | fused_reproject_surfaces | dropin_reproject_surfaces (temporal
    # reprojection onto the previous frame's surfaces: every rank gathers every slab's history and previous Visibility)
    mode = os.environ.get("SLAB_MODE", "fused")
    surfaces = mode.endswith("_reproject_surfaces")
    reproject = "surfaces" if surfaces else False
    fused = not mode.startswith("dropin")
    tris = small_scene("blocks_ao").copy()
    tris["emissive"][100:140] = (5.0, 4.0, 3.0)
    cam, W, H = ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0)), 320, 400
    if mode == "group":
        H = 800  # two slabs per GPU, each at least a halo tall
    if mode == "group":  # two slabs per GPU on two streams, linked by pointers within a process and by cudaIpc across
        part = slabs.SlabGroup(torch, dist, rank, world, tris, cam, W, H, sub=2)
    else:
        part = slabs.SlabRenderer(torch, dist, rank, world, tris, cam, W, H, fused=fused, p2p=(mode == "fused"),
                                  reproject=reproject)
    full = slabs.SlabRenderer(torch, None, 0, 1, tris, cam, W, H, fused=fused, reproject=reproject)
    for r in (part, full):
        r.set_reuse_weights(cedecrt.REUSE_UNBIASED)
    e, c = np.asarray(cam[0], np.float64), np.asarray(cam[1], np.float64)
    moves = {1: (tuple(e + (0.4, -0.2, 0.1)), tuple(c + (0.1, 0.0, -0.1))),
             2: (tuple(e + (0.9, -1.0, 0.3)), tuple(c + (0.2, 0.6, -0.2)))}
    for k in range(4):
        part.frame()
        full.frame()
        if k + 1 in moves:
            for s in part.slabs:
                s.set_camera(*moves[k + 1])
            full.set_camera(*moves[k + 1])
    for s in part.slabs:
        s.join()
    torch.cuda.synchronize()
    ok = True
    for sl in part.slabs:
        for name, elem in (("t_acc", 16), ("t_pix", 4), ("t_vis", 16)):
            a = sl._rows(getattr(sl, name), elem, sl.y0, sl.y1)
            b = full._rows(getattr(full, name), elem, sl.y0, sl.y1)
            ok = ok and bool(torch.equal(a, b))
    flags = [None] * world
    dist.all_gather_object(flags, ok)
    if rank == 0:
        print("GPU_SLABS_OK" if all(flags) else "GPU_SLABS_MISMATCH %s" % flags, "world", world, "mode", mode,
              "p2p", part.p2p, "edges", part.edges, flush=True)
    dist.barrier()
    part.close()
    dist.destroy_process_group()
    sys.exit(0 if all(flags) else 1)


if __name__ == "__main__":
    main()
